// wavefront.cu — see wavefront.cuh for the design.  Every arithmetic step is the same
// device code the megakernel uses (dev_intersect.cuh / dev_shade.cuh); only the order in
// which threads meet the work differs, so results are bit-identical between the two.
#include "wavefront.cuh"

#include <algorithm>

#include "dev_sample.cuh"

namespace mcskin {
MCSKIN_VARIANT_BEGIN

namespace {

constexpr int kWfThreads = 256;
// Minimum resident blocks per SM asked of the compiler (i.e. register caps), from sweeps on B200:
// 3 blocks (80 registers, no spills) for the trace kernel (at 64 registers it spills 116 bytes: -1.5 % frame
// rate), 4 blocks (64 registers) for the queued shade kernel, compiler's choice for the hard-shadow kernel and
// for the in-thread shadow form of the shade kernel.
#ifndef MCSKIN_WF_HIT0_MIN_BLOCKS
#define MCSKIN_WF_HIT0_MIN_BLOCKS 3
#endif
#ifndef MCSKIN_WF_SHADE_MIN_BLOCKS
#define MCSKIN_WF_SHADE_MIN_BLOCKS 4
#endif
#define WF_HIT0_BOUNDS __launch_bounds__(kWfThreads, MCSKIN_WF_HIT0_MIN_BLOCKS)
#ifdef MCSKIN_WF_SHADOW_MIN_BLOCKS
#define WF_SHADOW_BOUNDS __launch_bounds__(kWfThreads, MCSKIN_WF_SHADOW_MIN_BLOCKS)
#else
#define WF_SHADOW_BOUNDS __launch_bounds__(kWfThreads)
#endif
#define WF_SHADE_BOUNDS __launch_bounds__(kWfThreads, QUEUED ? MCSKIN_WF_SHADE_MIN_BLOCKS : 2)

// geo.w of a queue entry: box (16 bits) | face (3) | flip (1) | bounce depth (7; kMaxStackDepth = 64)
__device__ __forceinline__ unsigned int pack_hit(const Hit& h, int depth) {
    return static_cast<unsigned int>(h.box & 0xffff) | (static_cast<unsigned int>(h.face & 7) << 16) |
           (h.flip ? (1u << 19) : 0u) | (static_cast<unsigned int>(depth) << 20);
}
__device__ __forceinline__ int unpack_depth(float4 geo) { return static_cast<int>((__float_as_uint(geo.w) >> 20) & 0x7fu); }
__device__ __forceinline__ Hit unpack_hit(float4 geo, float4 org) {
    Hit h;
    const unsigned int k = __float_as_uint(geo.w);
    h.p = mk3(geo.x, geo.y, geo.z);
    h.box = static_cast<int>(k & 0xffffu);
    h.face = static_cast<int>((k >> 16) & 7u);
    h.flip = (k >> 19) & 1u;
    h.texel = __float_as_int(org.w);
    h.t = 0.0f;
    return h;
}
static_assert(kMaxStackDepth < 128, "the bounce depth of a queue entry has 7 bits");

// Appends the hits of a warp to the queue with one atomic; all 32 lanes must call.  Returns false for a
// lane whose hit found the queue full.
__device__ __forceinline__ bool enqueue_hit(const HitQueueView& q, unsigned int* counter, unsigned int capacity,
                                            bool isHit, const Hit& h, const Ray& ray, unsigned int path, int depth) {
    const unsigned int lane = threadIdx.x & 31u;
    const unsigned int m = __ballot_sync(0xffffffffu, isHit);
    if (m == 0u) return true;
    unsigned int base = 0u;
    if (lane == 0u) base = atomicAdd(counter, static_cast<unsigned int>(__popc(m)));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (isHit) {
        const unsigned int i = base + __popc(m & ((1u << lane) - 1u));
        if (i >= capacity) return false;
        q.geo[i] = make_float4(h.p.x, h.p.y, h.p.z, __uint_as_float(pack_hit(h, depth)));
        q.org[i] = make_float4(ray.o.x, ray.o.y, ray.o.z, __int_as_float(h.texel));
        q.dir[i] = make_float4(ray.d.x, ray.d.y, ray.d.z, __uint_as_float(path));
    }
    return true;
}


// ---------------------------------------------------------------- the paths' geometry
// Which surfaces a path meets does not depend on how they are shaded: the mirror ray of a hit is a
// function of the hit point, the normal and the incoming direction only (raytracer.cpp:133-140).  So one
// thread walks its sample's whole chain — primary ray, closest hit, mirror ray, closest hit, ... — and
// appends EVERY hit, tagged with its bounce depth, to the one hit queue.  The shadow and shading kernels
// then run once over all hits of all depths instead of once per depth: the frame has no chain of
// ever-shorter launches for the deeper bounces (they were a fifth of the frame time for a twentieth of
// its work).  How a chain ends is recorded here as well: a ray that leaves the scene fixes the path's
// terminal colour (gradient for camera rays, flat colour for mirror rays); a chain that reaches the
// bounce limit ends in a hit whose shaded colour the shading kernel stores as the terminal colour.
// The 32 samples of a warp belong to 32 / spp neighbouring pixels, so the lanes that bounce do so together.
constexpr int kPathOverflow = -2;  // top[path]: the queue was full; the path is redone in-thread (k_wf_overflow)

// AOV: also record every path's camera-ray hit for the AOV planes (aov_records; the normal and texel colour only when the
// frame has a guide plane, the texel index only when it has the texel plane).
template <bool BATCH, bool AOV>
__global__ void WF_HIT0_BOUNDS
k_wf_trace(const DevFrame fr, const FramePointers fp_, const ActiveList list_, const WaveView wv_, const AovView aov_,
           const AovView* __restrict__ aovBatch, const BatchSlice* __restrict__ batch) {
    __shared__ __align__(8) uint64_t stageBar;
    const FramePointers& fp = BATCH ? batch[blockIdx.y].fp : fp_;
    const ActiveList& list = BATCH ? batch[blockIdx.y].list : list_;
    const WaveView& wv = BATCH ? batch[blockIdx.y].wave : wv_;
    unsigned int count = *list.count;
    if (count > list.capacity) count = list.capacity;
    if (count > wv.slotCapacity) count = wv.slotCapacity;
    const unsigned long long nPaths = static_cast<unsigned long long>(count) * fr.spp;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * kWfThreads;
    if (static_cast<unsigned long long>(blockIdx.x) * kWfThreads >= nPaths) return;
    stage_bulk(g_sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(g_sceneSmem, fp.texels, fr);
    const int spp = fr.spp, dps = fr.draws_per_sample;
    const int lastBounce = min(fr.max_bounces, wv.levels);  // hits at this depth spawn no mirror ray

    for (unsigned long long p0 = static_cast<unsigned long long>(blockIdx.x) * kWfThreads + (threadIdx.x & ~31u);
         p0 < nPaths; p0 += stride) {
        const unsigned long long p = p0 + (threadIdx.x & 31u);
        bool alive = false;
        Hit hit;
        hit.box = -1; hit.face = 0; hit.texel = 0; hit.flip = false; hit.t = 0.0f; hit.p = mk3(0.f, 0.f, 0.f);
        Ray ray;
        ray.o = mk3(0.f, 0.f, 0.f);
        ray.d = mk3(0.f, 0.f, 0.f);
        if (p < nPaths) {
            const unsigned int slot = static_cast<unsigned int>(p / spp);
            const int s = static_cast<int>(p - static_cast<unsigned long long>(slot) * spp);
            const uint2 sp = list.slot_pixel[slot];
            if (sp.x != kUnusedSlot) {
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
                float u, v;
                sample_uv(fr, px, py, sd, &u, &v);
                ray = primary_ray(fr, u, v, sd);
                // (restricting this query to the boxes whose screen rectangle holds the pixel, as the primary
                // pass does, measured slower here: the branch-free reject pass over all boxes is cheaper than
                // the mask plus a bit loop when nearly every ray hits)
                hit = closest_hit(sc, ray);
                if (AOV) {
                    const AovView& av = BATCH ? aovBatch[blockIdx.y] : aov_;
                    const AovRecords rec = aov_records(wv, av.planes);
                    rec.t[p] = hit.t;
                    rec.id[p] = aov_id(hit);
                    if (aov_guides(av.planes) && hit.box >= 0) {
                        const V3 n = hit_normal(sc, hit);
                        rec.normal[p] = make_float4(n.x, n.y, n.z, 0.0f);
                        rec.albedo[p] = hit_texel(sc, hit);
                    }
                    if (av.planes.texel) rec.texel[p] = hit.texel;
                }
                if (fr.max_bounces < 0) {
                    // traceRay returns at once (depth 0 > maxBounces, raytracer.cpp:86-90); the tile
                    // renderer's re-test replaces misses by the gradient (tile_renderer.cpp:111-114)
                    wv.tail[p] = hit.box < 0 ? config_background(fr, u, v) : config_background(fr, 0.5f, 0.5f);
                    wv.top[p] = 0;
                } else if (hit.box < 0) {
                    wv.tail[p] = config_background(fr, u, v);
                    wv.top[p] = 0;
                } else {
                    alive = true;
                }
            } else {
                wv.top[p] = -1;  // unused slot
            }
        }
        // every live lane of the warp is at the same depth: they advance together
        for (int depth = 0; __any_sync(0xffffffffu, alive); ++depth) {
            const bool queued = enqueue_hit(wv.q, &wv.qCount[0], wv.qCapacity, alive, hit, ray, static_cast<unsigned int>(p), depth);
            if (!alive) continue;
            if (!queued) {
                wv.top[p] = kPathOverflow;
                alive = false;
            } else if (depth < lastBounce) {  // raytracer.cpp:133-140
                const V3 N = normalize3(hit_normal(sc, hit));
                const V3 D = normalize3(ray.d);
                V3 Rd = D - N * (2.0f * dot3(D, N));
                Rd = normalize3(Rd);
                ray.o = hit.p + N * kReflectEpsilon;
                ray.d = Rd;
                hit = closest_hit(sc, ray);
                if (hit.box < 0) {
                    wv.tail[p] = flat_background(fr);  // bounced rays see the flat colour (raytracer.cpp:101)
                    wv.top[p] = depth + 1;
                    alive = false;
                }
            } else {
                alive = false;  // the chain ends in this hit: k_wf_shade stores its colour as the terminal one
            }
        }
    }
}

// Paths whose hits did not fit the queue (only possible when the queue is smaller than
// paths x (bounces + 1), i.e. when the budget cut it): the whole path again, in one thread.
template <bool BATCH>
__global__ void __launch_bounds__(kWfThreads)
k_wf_overflow(const DevFrame fr, const FramePointers fp_, const ActiveList list_, const WaveView wv_,
              const BatchSlice* __restrict__ batch) {
    __shared__ __align__(8) uint64_t stageBar;
    const FramePointers& fp = BATCH ? batch[blockIdx.y].fp : fp_;
    const ActiveList& list = BATCH ? batch[blockIdx.y].list : list_;
    const WaveView& wv = BATCH ? batch[blockIdx.y].wave : wv_;
    if (wv.qCount[0] <= wv.qCapacity) return;  // nothing overflowed
    unsigned int count = *list.count;
    if (count > list.capacity) count = list.capacity;
    if (count > wv.slotCapacity) count = wv.slotCapacity;
    const unsigned long long nPaths = static_cast<unsigned long long>(count) * fr.spp;
    stage_bulk(g_sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(g_sceneSmem, fp.texels, fr);
    const int spp = fr.spp, dps = fr.draws_per_sample;
    for (unsigned long long p = static_cast<unsigned long long>(blockIdx.x) * kWfThreads + threadIdx.x; p < nPaths;
         p += static_cast<unsigned long long>(gridDim.x) * kWfThreads) {
        if (wv.top[p] != kPathOverflow) continue;
        const unsigned int slot = static_cast<unsigned int>(p / spp);
        const int s = static_cast<int>(p - static_cast<unsigned long long>(slot) * spp);
        const uint2 sp = list.slot_pixel[slot];
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
        wv.tail[p] = trace_path(sc, fr, primary_ray(fr, opt.u, opt.v, sd), opt);
        wv.top[p] = 0;
    }
}

// ---------------------------------------------------------------- soft shadows of every hit
// computeSoftShadow (shading.cpp:28-60) for every hit of the queue (all depths), in ONE kernel.  A block works through
// chunks of 256 hits, claimed from a device counter, in three block-synchronous phases:
//   A  thread = hit: the common origin of the hit's shadow rays and the boxes their bundle can reach.
//      Nothing in reach -> all N rays are lit by construction, the hit is done.  The others are
//      COMPACTED into a ring in shared memory, so that phase B runs with full warps however the
//      "nothing in reach" hits are spread over the queue (they were a third of the lanes of the
//      seeding loop when it ran per queue entry).
//   B  thread = pending hit, once 256 of them are waiting (or the queue is exhausted): the fresh
//      std::mt19937 of the hit (raytracer.cpp:110-113) — 396 dependent LCG steps — and its next
//      8 points on the light's disk, into shared memory.
//   C  thread = (pending hit, sample): one shadow ray; unoccluded rays are counted per hit.
// The light points never leave the SM (they were 96 B per hit written to and read back from HBM), and
// the engine runs only for hits that cast rays.  N > 8 samples: phases B and C repeat in rounds of 8,
// the engine state waiting in shared memory in between.
constexpr int kPendCap = 2 * kWfThreads;    // ring of hits waiting for their engine (power of two)
constexpr int kShadowRound = 8;             // light samples per hit and round
constexpr int kPtStride = kShadowRound * 3 + 1;  // floats per hit in the point table (odd: no bank conflicts)
struct ShadowSmem {
    float4 pendP[kPendCap];                 // hit point xyz, w = seed of the hit's engine (raytracer.cpp:110-112)
    float4 pendO[kPendCap];                 // shadow-ray origin xyz, w = box mask of the bundle
    unsigned int pendI[kPendCap];           // index in the queue
    float pts[kWfThreads * kPtStride];      // this round's sample points
    uint4 engine[kWfThreads];               // FreshStream between rounds (N > kShadowRound only)
    unsigned int lit[kWfThreads];
    unsigned int head, tail;                // monotonic: ring entries [head, tail) are pending
    unsigned int chunk;                     // the chunk claimed for this trip
};
static_assert((kPendCap & (kPendCap - 1)) == 0, "ring size must be a power of two");

#ifndef MCSKIN_WF_SOFT_MIN_BLOCKS
#define MCSKIN_WF_SOFT_MIN_BLOCKS 4
#endif
template <bool BATCH>
__global__ void __launch_bounds__(kWfThreads, MCSKIN_WF_SOFT_MIN_BLOCKS)
k_wf_softshadow(const DevFrame fr, const FramePointers fp_, const WaveView wv_, const BatchSlice* __restrict__ batch) {
    __shared__ __align__(8) uint64_t stageBar;
    const FramePointers& fp = BATCH ? batch[blockIdx.y].fp : fp_;
    const WaveView& wv = BATCH ? batch[blockIdx.y].wave : wv_;
    unsigned int n = wv.qCount[0];
    if (n > wv.qCapacity) n = wv.qCapacity;
    const unsigned int nChunks = (n + kWfThreads - 1) / kWfThreads;
    if (blockIdx.x >= nChunks) return;
    stage_bulk(g_sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(g_sceneSmem, fp.texels, fr);
    ShadowSmem* sm = reinterpret_cast<ShadowSmem*>(g_sceneSmem + ((fp.blob_bytes + 15u) & ~15u));
    const int tid = threadIdx.x, lane = tid & 31;
    const HitQueueView q = wv.q;
    const int N = fr.shadow_samples;
    const int rounds = (N + kShadowRound - 1) / kShadowRound;
    const V3 lightCentre = ld3(fr.light_pos);
    const uint32_t one = fr.spp > 0 ? 1u : 0u;  // a 1 the compiler cannot see through
    unsigned int* chunkCounter = wv.qCount + 1;
    if (tid == 0) {
        sm->head = 0u;
        sm->tail = 0u;
    }
    for (;;) {
        __syncthreads();
        if (tid == 0) sm->chunk = atomicAdd(chunkCounter, 1u);
        __syncthreads();
        const unsigned int c = sm->chunk;
        const bool last = c >= nChunks;  // the queue is exhausted: flush what is pending and leave
        if (!last) {  // ---- phase A
            const unsigned int i = c * kWfThreads + tid;
            bool pend = false;
            float4 eP = make_float4(0.f, 0.f, 0.f, 0.f), eO = eP;
            if (i < n) {
                const float4 g = q.geo[i];
                const Hit h = unpack_hit(g, make_float4(0.f, 0.f, 0.f, 0.f));
                // P + n*eps (isInShadow, shading.cpp:17); computeSoftShadow hands it the raw hit normal
                // (shading.cpp:54, raytracer.cpp:113)
                const V3 origin = h.p + hit_normal(sc, h) * kShadowEpsilon;
                const uint32_t allow = bundle_box_mask(sc, origin, lightCentre, fr.light_radius);
                if (allow == 0u && sc.n_boxes <= 32) {
                    wv.lit[i] = static_cast<unsigned int>(N);
                } else {
                    pend = true;
                    eP = make_float4(h.p.x, h.p.y, h.p.z, __uint_as_float(shadow_seed(h.p, unpack_depth(g))));
                    eO = make_float4(origin.x, origin.y, origin.z, __uint_as_float(allow));
                }
            }
            const unsigned int m = __ballot_sync(0xffffffffu, pend);
            if (m) {
                unsigned int base = 0u;
                if (lane == 0) base = atomicAdd(&sm->tail, static_cast<unsigned int>(__popc(m)));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (pend) {
                    const unsigned int pos = (base + __popc(m & ((1u << lane) - 1u))) & (kPendCap - 1);
                    sm->pendP[pos] = eP;
                    sm->pendO[pos] = eO;
                    sm->pendI[pos] = i;
                }
            }
            __syncthreads();
        }
        for (;;) {  // ---- drain the ring, 256 hits at a time
            const unsigned int head = sm->head;
            const unsigned int avail = sm->tail - head;
            if (avail == 0u || (!last && avail < static_cast<unsigned int>(kWfThreads))) break;
            const unsigned int cnt = avail < static_cast<unsigned int>(kWfThreads) ? avail : static_cast<unsigned int>(kWfThreads);
            const bool mine = static_cast<unsigned int>(tid) < cnt;
            if (mine) sm->lit[tid] = 0u;
            for (int round = 0; round < rounds; ++round) {
                const int ns = min(kShadowRound, N - round * kShadowRound);
                if (mine) {  // ---- phase B
                    const float4 eP = sm->pendP[(head + tid) & (kPendCap - 1)];
                    const V3 P = mk3(eP.x, eP.y, eP.z);
                    FreshStream rng;
                    if (round == 0) {
                        rng.seed_memo(__float_as_uint(eP.w), one, wv.seedMemo);
                    } else {
                        const uint4 e = sm->engine[tid];
                        rng.cur = e.x; rng.nxt = e.y; rng.far = e.z; rng.j = e.w;
                    }
                    soft_shadow_positions(fr, P, ns, rng, sm->pts + tid * kPtStride);
                    if (round + 1 < rounds) sm->engine[tid] = make_uint4(rng.cur, rng.nxt, rng.far, rng.j);
                }
                __syncthreads();
                const unsigned int nRays = cnt * static_cast<unsigned int>(ns);  // ---- phase C
                for (unsigned int r = tid; r < nRays; r += kWfThreads) {
                    const unsigned int e = ns == kShadowRound ? r >> 3 : r / static_cast<unsigned int>(ns);
                    const unsigned int k = r - e * static_cast<unsigned int>(ns);
                    const float4 eO = sm->pendO[(head + e) & (kPendCap - 1)];
                    const float* pt = sm->pts + e * kPtStride + k * 3u;
                    if (!in_shadow_from(sc, mk3(eO.x, eO.y, eO.z), mk3(pt[0], pt[1], pt[2]), __float_as_uint(eO.w)))
                        atomicAdd(&sm->lit[e], 1u);
                }
                __syncthreads();
            }
            if (mine) wv.lit[sm->pendI[(head + tid) & (kPendCap - 1)]] = sm->lit[tid];
            __syncthreads();
            if (tid == 0) sm->head = head + cnt;
            __syncthreads();
        }
        if (last) break;
    }
}

// hard shadows: one ray from every hit to the light's centre (isInShadow as shade() calls it, with the
// normalised normal: shading.cpp:69,78)
template <bool BATCH>
__global__ void __launch_bounds__(kWfThreads)
k_wf_hardshadow(const DevFrame fr, const FramePointers fp_, const WaveView wv_, const BatchSlice* __restrict__ batch) {
    __shared__ __align__(8) uint64_t stageBar;
    const FramePointers& fp = BATCH ? batch[blockIdx.y].fp : fp_;
    const WaveView& wv = BATCH ? batch[blockIdx.y].wave : wv_;
    unsigned int n = wv.qCount[0];
    if (n > wv.qCapacity) n = wv.qCapacity;
    if (blockIdx.x * kWfThreads >= n) return;
    stage_bulk(g_sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(g_sceneSmem, fp.texels, fr);
    const HitQueueView q = wv.q;
    const V3 lightCentre = ld3(fr.light_pos);
    for (unsigned int i = blockIdx.x * kWfThreads + threadIdx.x; i < n; i += gridDim.x * kWfThreads) {
        const Hit h = unpack_hit(q.geo[i], make_float4(0.f, 0.f, 0.f, 0.f));
        // (a box mask for the single ray, as for soft-shadow bundles, costs more than the one ray it can save)
        wv.lit[i] = in_shadow(sc, h.p, normalize3(hit_normal(sc, h)), lightCentre) ? 0u : 1u;
    }
}

// ---------------------------------------------------------------- shading
// shade() for every hit of the queue (shading.cpp:62-96 + raytracer.cpp:116-131): Blinn-Phong with the
// visibility the shadow kernel counted, ambient occlusion for camera-ray hits.  A hit that spawned a mirror
// ray stores its colour on the path's bounce stack; the last hit of a chain that reached the bounce limit
// stores the path's terminal colour.
// QUEUED: the visibility comes from the shadow kernel's counters; otherwise (rare shadow settings: N > 113,
// N <= 1, a point light) shadows are evaluated in place.
template <bool QUEUED, bool BATCH>
__global__ void WF_SHADE_BOUNDS
k_wf_shade(const DevFrame fr, const FramePointers fp_, const WaveView wv_, const BatchSlice* __restrict__ batch) {
    const FramePointers& fp = BATCH ? batch[blockIdx.y].fp : fp_;
    const WaveView& wv = BATCH ? batch[blockIdx.y].wave : wv_;
    __shared__ __align__(8) uint64_t stageBar;
    unsigned int n = wv.qCount[0];
    if (n > wv.qCapacity) n = wv.qCapacity;
    if (blockIdx.x * kWfThreads >= n) return;
    stage_bulk(g_sceneSmem, fp.blob, fp.blob_bytes, &stageBar);
    const SceneView sc = scene_view(g_sceneSmem, fp.texels, fr);
    const HitQueueView q = wv.q;
    const bool cfg = fr.use_config != 0;
    const size_t cap = wv.pathCapacity;
    const int lastBounce = min(fr.max_bounces, wv.levels);

    for (unsigned int i = blockIdx.x * kWfThreads + threadIdx.x; i < n; i += gridDim.x * kWfThreads) {
        const float4 g = q.geo[i], o = q.org[i], dd = q.dir[i];
        const Hit h = unpack_hit(g, o);
        const int d = unpack_depth(g);
        const unsigned int path = __float_as_uint(dd.w);
        const V3 P = h.p;
        const V3 nrm = hit_normal(sc, h);
        const float4 tex = hit_texel(sc, h);
        const V3 viewDir = normalize3(mk3(o.x, o.y, o.z) - P);
        float vis;
        if (QUEUED) {
            vis = static_cast<float>(wv.lit[i]) / static_cast<float>(wv.shadowRays);
            if (wv.shadowMode == kShadowHard) vis = wv.lit[i] ? 1.0f : 0.0f;
        } else if (cfg && fr.soft_on) {
            vis = soft_shadow(sc, fr, P, nrm, fr.shadow_samples, shadow_seed(P, d));
        } else {
            vis = in_shadow(sc, P, normalize3(nrm), ld3(fr.light_pos)) ? 0.0f : 1.0f;
        }
        float4 shaded = shade_lit(fr, P, nrm, tex, viewDir, vis);
        const float alpha = shaded.w;
        if (cfg && fr.ao_on && d == 0) {
            const float ao = ambient_occlusion(sc, P, nrm, fr.ao_samples, fr.ao_radius, ao_seed(P));
            const float f = 1.0f - fr.ao_intensity * (1.0f - ao);
            shaded.x *= f;
            shaded.y *= f;
            shaded.z *= f;
        }
        if (d < lastBounce) {
            wv.stack[static_cast<size_t>(d) * cap + path] = make_float4(shaded.x, shaded.y, shaded.z, alpha);
        } else {
            shaded.w = alpha;
            wv.tail[path] = clamp4(shaded);
            wv.top[path] = d;
        }
    }
}

// ---------------------------------------------------------------- fold + ordered average
__device__ __forceinline__ float4 fold_path(const WaveView& wv, size_t path) {
    float4 c = wv.tail[path];
    const int top = wv.top[path];
    if (top > 0) {
        const size_t cap = wv.pathCapacity;
        const float alpha0 = wv.stack[path].w;
        const float keep = 1.0f - kReflectivity;
        for (int k = top - 1; k >= 0; --k) {  // raytracer.cpp:143-147, innermost level first
            const float4 s = wv.stack[static_cast<size_t>(k) * cap + path];
            float4 m;
            m.x = s.x * keep + c.x * kReflectivity;
            m.y = s.y * keep + c.y * kReflectivity;
            m.z = s.z * keep + c.z * kReflectivity;
            m.w = alpha0;
            c = clamp4(m);
        }
    }
    return c;
}

// The AOV planes of the pixel whose spp paths start at path0, from the paths' records (k_wf_trace), in sample order.
__device__ __forceinline__ void fold_aov(const DevFrame& fr, const McAovTargets& planes, const AovRecords& rec, size_t path0,
                                         int spp, unsigned int pixelIndex) {
    AovFold a;
    for (int i = 0; i < spp; ++i) a.add(rec.t[path0 + i], rec.id[path0 + i]);
    store_aov(fr, planes, pixelIndex, a);
    if (planes.texel) {
        int texel = -1;
        for (int i = 0; i < spp; ++i)
            if (rec.id[path0 + i] >= 0) {
                texel = rec.texel[path0 + i];
                break;
            }
        store_texel(planes, pixelIndex, texel);
    }
    if (!aov_guides(planes)) return;
    GuideFold g;
    for (int i = 0; i < spp; ++i)
        if (rec.id[path0 + i] >= 0) g.add(rec.normal[path0 + i], rec.albedo[path0 + i]);
    store_guides(planes, pixelIndex, a.n, g);
}

// FAR: the form for images across a link (BandView::far_output); two instantiations, so that the streaming form keeps
// its 32 registers (8 resident blocks: the kernel lives on loads in flight).
// AOV: the first lane of every pixel also folds the pixel's recorded camera-ray hits in sample order (store_aov,
// store_texel, store_guides).
template <bool BATCH, bool FAR, bool AOV>
__global__ void __launch_bounds__(kWfThreads)
k_wf_resolve_warp(const DevFrame fr, const BandView band_, const ActiveList list_, const WaveView wv_, const int lgSpp,
                  const AovView aov_, const AovView* __restrict__ aovBatch, const BatchSlice* __restrict__ batch) {
    const BandView band = hot_band(BATCH ? batch[blockIdx.y].band : band_);  // listed pixels lie in tiles the figure's rectangle touches
    const ActiveList& list = BATCH ? batch[blockIdx.y].list : list_;
    const WaveView& wv = BATCH ? batch[blockIdx.y].wave : wv_;
    __shared__ __align__(16) float stageAll[kWfThreads / 32][kWarpStageFloats];
    __shared__ __align__(16) float4 outAll[FAR ? kWfThreads / 32 : 1][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned int count = *list.count;
    if (!BATCH && list.count_host && blockIdx.x == 0 && threadIdx.x == 0) *list.count_host = count;  // for the statistics
    if (count > list.capacity) count = list.capacity;
    if (count > wv.slotCapacity) count = wv.slotCapacity;
    const int spp = fr.spp;
    const int pixPerGroup = 32 >> lgSpp;
    const int pix = lane >> lgSpp, s = lane & (spp - 1);
    float* stageW = stageAll[warp];
    float4* outW = outAll[FAR ? warp : 0];
    // One round: the 32 samples of 32 / spp listed pixels (slot = firstSlot + pix for this lane), folded and averaged in
    // sample order; the averages go to the image, or to outStage for the caller to store.
    auto round = [&](unsigned int slot, unsigned int pixelIndex, float4* outStage) {
        const bool on = pixelIndex != kUnusedSlot;
        float4 colour = make_float4(0.f, 0.f, 0.f, 0.f);
        if (on) colour = fold_path(wv, static_cast<size_t>(slot) * spp + s);
        const unsigned int leaders = __ballot_sync(0xffffffffu, on && s == 0);
        unsigned int resolveMask = 0u;
        unsigned int m = leaders;
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1u;
            resolveMask |= 1u << (l >> lgSpp);
        }
        warp_resolve<true>(fr, band, stageW, lane, spp, lgSpp, colour, pixelIndex, resolveMask, outStage);
        if (AOV && on && s == 0) {
            const AovView& av = BATCH ? aovBatch[blockIdx.y] : aov_;
            fold_aov(fr, av.planes, aov_records(wv, av.planes), static_cast<size_t>(slot) * spp, spp, pixelIndex);
        }
    };
    if (!FAR) {
        // the image is this device's memory: rounds dealt to the warps of the grid in turn (the grid streams through the
        // path arrays front to back), every pixel stored as soon as it is averaged
        const unsigned int nRounds = (count + pixPerGroup - 1) / pixPerGroup;
        for (unsigned int g = blockIdx.x * (kWfThreads / 32) + warp; g < nRounds; g += gridDim.x * (kWfThreads / 32)) {
            const unsigned int slot = g * pixPerGroup + pix;
            round(slot, slot < count ? list.slot_pixel[slot].x : kUnusedSlot, nullptr);
        }
        return;
    }
    // The image lies across PCIe or NVLink (a mapped host image, a peer's frame): stores of 16 bytes at a time waste the
    // link.  Every warp takes an equal run of consecutive slots — the primary pass hands out slots in runs of
    // neighbouring pixels of a tile row — and works through it up to 32 slots at a time: the rounds' averages go to
    // shared memory, then lane l stores pixel l, so neighbours leave as one piece of up to 512 bytes.  Equal runs,
    // because the rounds of a warp are dependent loads in series and a frame has only some ten of them per warp.
    const unsigned int totalWarps = gridDim.x * (kWfThreads / 32);
    const unsigned int perWarp = ((count + totalWarps - 1u) / totalWarps + pixPerGroup - 1u) / pixPerGroup * pixPerGroup;
    const unsigned int first = (blockIdx.x * (kWfThreads / 32) + warp) * perWarp;
    const unsigned int last = min(count, first + perWarp);
    for (unsigned int base = first; base < last; base += 32u) {
        const unsigned int mySlot = base + lane;
        const unsigned int myPixel = mySlot < last ? list.slot_pixel[mySlot].x : kUnusedSlot;
        const int rounds = (static_cast<int>(min(32u, last - base)) + pixPerGroup - 1) >> (5 - lgSpp);
        for (int g = 0; g < rounds; ++g) {
            const int local = g * pixPerGroup + pix;  // slot of the batch this lane's sample belongs to
            const unsigned int pixelIndex = __shfl_sync(0xffffffffu, myPixel, local);
            if (__ballot_sync(0xffffffffu, pixelIndex != kUnusedSlot) == 0u) continue;
            round(base + local, pixelIndex, outW + g * pixPerGroup);
        }
        __syncwarp();
        if (myPixel != kUnusedSlot) store_pixel(band, myPixel, outW[lane]);  // (outW: warp_resolve<true> output)
        __syncwarp();
    }
}

// any spp: one thread sums a pixel's folded samples in order
template <bool BATCH, bool AOV>
__global__ void __launch_bounds__(kWfThreads)
k_wf_resolve_pixel(const DevFrame fr, const BandView band_, const ActiveList list_, const WaveView wv_,
                   const AovView aov_, const AovView* __restrict__ aovBatch, const BatchSlice* __restrict__ batch) {
    const BandView band = hot_band(BATCH ? batch[blockIdx.y].band : band_);
    const ActiveList& list = BATCH ? batch[blockIdx.y].list : list_;
    const WaveView& wv = BATCH ? batch[blockIdx.y].wave : wv_;
    unsigned int count = *list.count;
    if (!BATCH && list.count_host && blockIdx.x == 0 && threadIdx.x == 0) *list.count_host = count;  // for the statistics
    if (count > list.capacity) count = list.capacity;
    if (count > wv.slotCapacity) count = wv.slotCapacity;
    const int spp = fr.spp;
    for (unsigned int slot = blockIdx.x * kWfThreads + threadIdx.x; slot < count; slot += gridDim.x * kWfThreads) {
        const uint2 sp = list.slot_pixel[slot];
        if (sp.x == kUnusedSlot) continue;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int s = 0; s < spp; ++s) acc = add4(acc, fold_path(wv, static_cast<size_t>(slot) * spp + s));
        store_shaded_pixel(band, sp.x, scale4(acc, fr.inv_spp));
        if (AOV) {
            const AovView& av = BATCH ? aovBatch[blockIdx.y] : aov_;
            fold_aov(fr, av.planes, aov_records(wv, av.planes), static_cast<size_t>(slot) * spp, spp, sp.x);
        }
    }
}

// zeroes the active-pixel counter and the queue counters of every scene of a batch
__global__ void k_batch_reset(const BatchSlice* __restrict__ batch, const int nScenes, const int nQueueCounters) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nScenes) return;
    *batch[s].list.count = 0u;
    for (int i = 0; i < nQueueCounters; ++i) batch[s].wave.qCount[i] = 0u;
}

int log2_pow2_le32(int v) {
    for (int lg = 0; lg <= 5; ++lg)
        if (v == (1 << lg)) return lg;
    return -1;
}

size_t align256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

int shadow_mode_of(const DevFrame& fr) {
    if (!(fr.use_config && fr.soft_on)) return kShadowHard;
    if (fr.shadow_samples <= 1 || fr.light_radius < 1e-4f || 2 * fr.shadow_samples > kFreshStreamMaxDraws)
        return kShadowInThread;
    return kShadowSoft;
}
int stack_levels_of(const DevFrame& fr) {
    return fr.max_bounces < 0 ? 0 : (fr.max_bounces > kMaxStackDepth ? kMaxStackDepth : fr.max_bounces);
}
constexpr size_t kEntryBytes = 3 * sizeof(float4) + sizeof(unsigned int);  // geo, org, dir, lit
constexpr int kQueueCounters = 4;

}  // namespace

int wavefront_max_hits_per_path(const DevFrame& fr) { return stack_levels_of(fr) + 1; }
size_t wavefront_bytes_per_path(const DevFrame& fr, bool aov, bool guides, bool texel) {
    // tail, top, bounce stack (+ the camera ray's hit distance and id, + its normal and texel colour, + its texel index)
    return sizeof(float4) + sizeof(int) + sizeof(float4) * stack_levels_of(fr) + (aov ? sizeof(float) + sizeof(int) : 0) +
           (aov && guides ? 2 * sizeof(float4) : 0) + (aov && texel ? sizeof(int) : 0);
}
size_t wavefront_bytes_per_entry() { return kEntryBytes; }
size_t wavefront_fixed_bytes(const DevFrame&) { return 256 * 16 + sizeof(unsigned int) * kQueueCounters; }

bool wavefront_carve(const DevFrame& fr, void* base, size_t bytes, unsigned int pathCapacity, unsigned int entryCapacity,
                     int gridBlocks, WaveView* out, const McAovTargets* aov) {
    WaveView w{};
    w.pathCapacity = pathCapacity;
    w.slotCapacity = pathCapacity / static_cast<unsigned int>(fr.spp);
    w.qCapacity = entryCapacity;
    w.levels = stack_levels_of(fr);
    w.shadowMode = shadow_mode_of(fr);
    w.shadowRays = w.shadowMode == kShadowSoft ? fr.shadow_samples : (w.shadowMode == kShadowHard ? 1 : 0);
    w.gridBlocks = gridBlocks;
    w.softGrid = gridBlocks;
    unsigned char* p = static_cast<unsigned char*>(base);
    size_t off = 0;
    auto take = [&](size_t n) {
        void* r = p + off;
        off = align256(off + n);
        return r;
    };
    const size_t cap = pathCapacity, ents = entryCapacity;
    w.q.geo = static_cast<float4*>(take(ents * sizeof(float4)));
    w.q.org = static_cast<float4*>(take(ents * sizeof(float4)));
    w.q.dir = static_cast<float4*>(take(ents * sizeof(float4)));
    w.lit = static_cast<unsigned int*>(take(ents * sizeof(unsigned int)));
    w.tail = static_cast<float4*>(take(cap * sizeof(float4)));
    w.top = static_cast<int*>(take(cap * sizeof(int)));
    w.stack = static_cast<float4*>(take(std::max<size_t>(16, cap * sizeof(float4) * w.levels)));
    // [0] hits in the queue (counts on beyond the capacity: overflow), [1] chunk counter of the soft-shadow kernel
    w.qCount = static_cast<unsigned int*>(take(sizeof(unsigned int) * kQueueCounters));
    if (aov) {  // in aov_records' order, right after the counters
        if (take(cap * sizeof(float)) != aov_records(w, *aov).t) return false;
        take(cap * sizeof(int));
        if (aov_guides(*aov)) {
            take(cap * sizeof(float4));
            take(cap * sizeof(float4));
        }
        if (aov->texel) take(cap * sizeof(int));
    }
    if (off > bytes) return false;
    *out = w;
    return true;
}

void launch_batch_reset(const BatchSlice* batch, int nScenes, cudaStream_t stream) {
    if (nScenes > 0) k_batch_reset<<<(nScenes + 127) / 128, 128, 0, stream>>>(batch, nScenes, kQueueCounters);
}

void launch_wavefront(const DevFrame& fr, const FramePointers& fp, const BandView& band, const ActiveList& list,
                      const WaveView& wv, unsigned int* groupCounter, cudaStream_t stream, int* launches,
                      const BatchSlice* batch, int nScenes, const AovView* aovView, const AovView* aovBatch) {
    int n = 0;
    const AovView av = aovView ? *aovView : AovView{};
    const int grid = wv.gridBlocks;
    const unsigned int ny = batch ? static_cast<unsigned int>(nScenes) : 1u;
    const dim3 g(grid, ny);
    const size_t blob = fp.blob_bytes;
#define MCSKIN_WF_LAUNCH(KERNEL, GRID, SMEM, ...)                                                   \
    do {                                                                                            \
        if (batch) KERNEL<true><<<GRID, kWfThreads, SMEM, stream>>>(__VA_ARGS__, batch);            \
        else KERNEL<false><<<GRID, kWfThreads, SMEM, stream>>>(__VA_ARGS__, batch);                 \
        ++n;                                                                                        \
    } while (0)
    if (wv.shadowMode == kShadowSoft) {  // ring + point table + scene blob exceed the default 48 KB
        static SmemOptIn optIn;
        static const void* const fns[] = {reinterpret_cast<const void*>(k_wf_softshadow<false>),
                                          reinterpret_cast<const void*>(k_wf_softshadow<true>)};
        optIn.limit(fns, 2);
    }
    // a batch's queue counters are zeroed by the caller (one kernel over all scenes)
    if (!batch) cudaMemsetAsync(wv.qCount, 0, sizeof(unsigned int) * kQueueCounters, stream);
    // every hit of every path, all bounce depths, into the one queue
    const bool aov = batch ? aovBatch != nullptr : aov_any(&av.planes);
    if (batch) {
        if (aov) k_wf_trace<true, true><<<g, kWfThreads, blob, stream>>>(fr, fp, list, wv, av, aovBatch, batch);
        else k_wf_trace<true, false><<<g, kWfThreads, blob, stream>>>(fr, fp, list, wv, av, aovBatch, batch);
    } else {
        if (aov) k_wf_trace<false, true><<<g, kWfThreads, blob, stream>>>(fr, fp, list, wv, av, aovBatch, batch);
        else k_wf_trace<false, false><<<g, kWfThreads, blob, stream>>>(fr, fp, list, wv, av, aovBatch, batch);
    }
    ++n;
    if (fr.max_bounces >= 0) {
        if (wv.shadowMode == kShadowSoft) {
            // persistent blocks that claim chunks of 256 hits: no more of them than can be resident
            const dim3 gs(std::max(1, std::min<int>(grid, wv.softGrid)), ny);
            const size_t smem = ((blob + 15u) & ~size_t(15)) + sizeof(ShadowSmem);
            MCSKIN_WF_LAUNCH(k_wf_softshadow, gs, smem, fr, fp, wv);
        } else if (wv.shadowMode == kShadowHard) {
            MCSKIN_WF_LAUNCH(k_wf_hardshadow, g, blob, fr, fp, wv);
        }
        if (wv.shadowMode != kShadowInThread) {
            if (batch) k_wf_shade<true, true><<<g, kWfThreads, blob, stream>>>(fr, fp, wv, batch);
            else k_wf_shade<true, false><<<g, kWfThreads, blob, stream>>>(fr, fp, wv, batch);
        } else {
            if (batch) k_wf_shade<false, true><<<g, kWfThreads, blob, stream>>>(fr, fp, wv, batch);
            else k_wf_shade<false, false><<<g, kWfThreads, blob, stream>>>(fr, fp, wv, batch);
        }
        ++n;
        // only a queue smaller than paths x (bounces + 1) can overflow
        if (static_cast<unsigned long long>(wv.qCapacity) < static_cast<unsigned long long>(wv.pathCapacity) * (wv.levels + 1))
            MCSKIN_WF_LAUNCH(k_wf_overflow, g, blob, fr, fp, list, wv);
    }
    const int lg = log2_pow2_le32(fr.spp);
    if (lg >= 0) {
        const bool farImage = !batch && band.far_output != 0;
        if (aov) {
            if (batch) k_wf_resolve_warp<true, false, true><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, lg, av, aovBatch, batch);
            else if (farImage) k_wf_resolve_warp<false, true, true><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, lg, av, aovBatch, batch);
            else k_wf_resolve_warp<false, false, true><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, lg, av, aovBatch, batch);
        } else {
            if (batch) k_wf_resolve_warp<true, false, false><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, lg, av, aovBatch, batch);
            else if (farImage) k_wf_resolve_warp<false, true, false><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, lg, av, aovBatch, batch);
            else k_wf_resolve_warp<false, false, false><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, lg, av, aovBatch, batch);
        }
        ++n;
    } else {
        if (batch && aov) k_wf_resolve_pixel<true, true><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, av, aovBatch, batch);
        else if (batch) k_wf_resolve_pixel<true, false><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, av, aovBatch, batch);
        else if (aov) k_wf_resolve_pixel<false, true><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, av, aovBatch, batch);
        else k_wf_resolve_pixel<false, false><<<g, kWfThreads, 0, stream>>>(fr, band, list, wv, av, aovBatch, batch);
        ++n;
    }
#undef MCSKIN_WF_LAUNCH
    // pixels the queues could not take: megakernel, starting at the first slot beyond them
    // (never in a batch: its queues are sized for every pixel of a scene)
    if (!batch && wv.slotCapacity < list.capacity) {
        n += MCSKIN_VARIANT_NS::launch_shade(fr, fp, band, list, grid, groupCounter, wv.slotCapacity, stream, 1, aov ? &av.planes : nullptr);  // (this build's)
    }
    if (launches) *launches += n;
}

MCSKIN_VARIANT_END
}  // namespace mcskin
