// wavefront.cuh — the shading pass as a wavefront of small kernels.
//
// The megakernel (one thread walks one sample through hit -> 8 shadow rays -> shade ->
// bounce -> ...) measured at half the issue rate of the chip: ncu showed warps waiting for
// instructions (a 275 KB program whose live part does not fit the instruction cache once
// warps drift apart) and, when they were kept together with block barriers, waiting for the
// slowest warp of the block.  The wavefront form runs the same arithmetic as a sequence of
// short, uniform kernels over compact queues in HBM:
//
//   k_wf_trace   thread = sample of a listed pixel: primary ray, closest hit, mirror ray, closest hit, ...
//                The chain a path follows does not depend on shading, so the whole of it is walked here and
//                EVERY hit, tagged with its bounce depth, goes into the one hit queue; a ray that leaves the
//                scene fixes the path's terminal colour (gradient for camera rays, flat colour for mirror rays)
//   k_wf_softshadow  block = chunks of 256 hits (all depths): the boxes each hit's shadow-ray bundle can reach;
//                hits that reach none are lit; the others are compacted in shared memory, get their fresh
//                std::mt19937 (397-step seeding) and the N points on the light's disk computeSoftShadow
//                would sample, then one thread per (hit, sample) casts the ray
//                (k_wf_hardshadow with soft shadows off: one ray per hit to the light's centre)
//   k_wf_shade   thread = hit: Blinn-Phong with the counted visibility, AO -> the path's bounce stack,
//                or its terminal colour if the chain ends in this hit
//   k_wf_resolve thread = sample: folds the bounce chain back to front with the reference's
//                mix, then the ordered per-pixel average.
// Five launches per frame whatever the bounce limit: the deeper bounces, a twentieth of the work, used to be a
// chain of ever-shorter launches per depth that took a fifth of the frame time (and nearly half of one GPU's
// share of a frame split eight ways).
//
// Every kernel is a persistent grid-stride loop over a device-side count, so nothing is
// read back to the host between them.  Pixels beyond the path capacity (extreme close-ups) are shaded by
// the megakernel instead, and paths whose hits do not fit a budget-limited queue are redone in one thread
// (k_wf_overflow); results are identical either way.
#pragma once
#include "kernels.cuh"

namespace mcskin {

struct HitQueueView {
    float4* geo;  // hit point xyz, w = box | face << 16 | flip << 19 | bounce depth << 20
    float4* org;  // ray origin xyz, w = texel index
    float4* dir;  // ray direction xyz, w = path index
};

struct WaveView {
    HitQueueView q;          // every hit of every path, all bounce depths
    unsigned int* lit;       // per queue entry: unoccluded shadow rays
    float4* tail;            // per path: colour returned by the deepest traceRay call
    float4* stack;           // [level][path]: shaded colour of every level that spawned a reflection (w = its alpha)
    int* top;                // per path: number of stack levels in use (-1: unused slot, -2: queue overflow)
    unsigned int* qCount;    // [0] hits appended to the queue (keeps counting beyond qCapacity), [1] chunk counter of
                             // the soft-shadow kernel; zeroed before the frame
    unsigned int pathCapacity;
    unsigned int slotCapacity;  // pixels handled by the wavefront = pathCapacity / spp
    unsigned int qCapacity;  // queue entries; paths x (levels + 1) can never overflow
    int levels;              // stack levels allocated = bounce depths traced
    int shadowMode;          // see enum below
    int shadowRays;          // rays per hit cast by the shadow kernel
    int gridBlocks;
    int softGrid;            // blocks of the soft-shadow kernel (persistent: what fits the device at once)
    uint2* seedMemo;         // FreshStream::seed_memo's table (kSeedMemoEntries entries), or null
};

// The AOV planes of a frame (or of one scene of a batch).  Kept apart from WaveView and BatchSlice: the batched kernels
// index a BatchSlice array, whose 256-byte stride is a shift.  The wavefront's per-path records of the planes lie in
// the WaveView's buffer (aov_records): the wavefront kernels take an AovView by value, and one that holds nothing but
// the planes keeps the parameters of the kernels of frames without planes as they are.
struct AovView {
    McAovTargets planes;
};

// Per path, the camera ray's closest hit as the planes need it, written by k_wf_trace and folded per pixel by the
// resolve kernels: distance and McHit-style id (-1: miss); for the guide planes also McHit.normal (xyz) and
// McHit.tex_color, for hits only.  wavefront_carve puts them right after the queue counters, in this order, each
// array 256-byte aligned.
struct AovRecords {
    float* t;
    int* id;
    float4* normal;
    float4* albedo;
};
__host__ __device__ inline size_t aov_align256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }
__host__ __device__ inline AovRecords aov_records(const WaveView& wv) {
    unsigned char* const base = reinterpret_cast<unsigned char*>(wv.qCount) + 256;  // (the counters take 16 bytes)
    const size_t cap = wv.pathCapacity;
    AovRecords r;
    r.t = reinterpret_cast<float*>(base);
    r.id = reinterpret_cast<int*>(base + aov_align256(cap * sizeof(float)));
    r.normal = reinterpret_cast<float4*>(base + 2 * aov_align256(cap * sizeof(float)));
    r.albedo = r.normal + aov_align256(cap * sizeof(float4)) / sizeof(float4);
    return r;
}

enum : int {
    kShadowHard = 0,      // no soft shadows: one ray to the light centre, normalised normal (shade())
    kShadowSoft = 1,      // computeSoftShadow with 2 <= N <= 113 samples: seed + N rays per hit
    kShadowInThread = 2   // rare forms (N > 113, N <= 1, radius < 1e-4): evaluated inside k_wf_shade
};

// One scene of a batched launch (SURVEY.md §8e: many skins per launch).  Scenes that share a frame
// description (image size, sampling, camera, light, box layout) are rendered by the same launches:
// blockIdx.y picks the scene, and with it the scene's boxes and texels, its output image, its work
// list and its queues.  A null batch pointer means the single scene passed by value.
struct BatchSlice {
    FramePointers fp;
    BandView band;
    ActiveList list;
    WaveView wave;
};
static_assert(sizeof(BatchSlice) == 256, "a BatchSlice is indexed by blockIdx.y: keep its stride a power of two");

// Storage: per path (terminal colour, stack height, bounce stack), per queue entry (hit record + lit counter).
// aov: the frame writes AOV planes (8 more bytes per path); guides: normal or albedo among them (32 more).
size_t wavefront_bytes_per_path(const DevFrame& fr, bool aov = false, bool guides = false);
size_t wavefront_bytes_per_entry();
size_t wavefront_fixed_bytes(const DevFrame& fr);
// Hits a path can put into the queue: bounce levels + 1.  A queue of pathCapacity times this cannot overflow.
int wavefront_max_hits_per_path(const DevFrame& fr);
// Carves the views out of one allocation of at least pathCapacity * wavefront_bytes_per_path +
// entryCapacity * wavefront_bytes_per_entry + wavefront_fixed_bytes (+ 256 per array) bytes; false if too small.
// aov (frames with AOV planes): also carves the per-path records these planes need (aov_records).
bool wavefront_carve(const DevFrame& fr, void* base, size_t bytes, unsigned int pathCapacity, unsigned int entryCapacity,
                     int gridBlocks, WaveView* out, const McAovTargets* aov = nullptr);

// The AOV defaults (coverage 0, depth 0, tri_id -1, normal and albedo zeros) into every pixel of the band's tiles (of every scene of a batch), before
// the primary pass; the shading pass then overwrites the pixels it resolves.  Only for bands with AOV planes.
// aovBatch: the device array of a batch's per-scene AOV views (null: one frame, `planes`).
void launch_aov_defaults(const DevFrame& fr, const BandView& band, const McAovTargets& planes, const AovView* aovBatch, int nScenes,
                         cudaStream_t stream);

// Shades every listed pixel (slots < wave.slotCapacity through the wavefront, the rest through the
// megakernel) and writes the band image.  groupCounter: zeroed device counter.
// batch / nScenes: device array of per-scene slices and its length (launches get gridDim.y = nScenes);
// every slice must have slotCapacity >= its list's capacity (no megakernel overflow in batches).
// aov / aovBatch: the frame's AOV view, or the device array of a batch's per-scene views (null: no AOV planes).
// launch_primary_batch: the primary pass over the scenes of a batch (pixel-per-lane kernels only): returns false if the
// frame description needs one of the other primary kernels, which have no batched form.
// (declared for both builds of the kernels: dev_types.cuh)
#define MCSKIN_HOT_WAVEFRONT_LAUNCHERS                                                                                   \
    void launch_wavefront(const DevFrame& fr, const FramePointers& fp, const BandView& band, const ActiveList& list,    \
                          const WaveView& wave, unsigned int* groupCounter, cudaStream_t stream, int* launches,         \
                          const BatchSlice* batch = nullptr, int nScenes = 1, const AovView* aov = nullptr,             \
                          const AovView* aovBatch = nullptr);                                                          \
    void launch_batch_reset(const BatchSlice* batch, int nScenes, cudaStream_t stream);                                 \
    bool launch_primary_batch(const DevFrame& fr, const BandView& band, uint32_t* tileStates, bool seedTiles,           \
                              const BatchSlice* batch, int nScenes, unsigned int blobBytes, int primaryTargetBlocks,    \
                              cudaStream_t stream);
MCSKIN_HOT_WAVEFRONT_LAUNCHERS
namespace plain {
MCSKIN_HOT_WAVEFRONT_LAUNCHERS
}
namespace counter {
MCSKIN_HOT_WAVEFRONT_LAUNCHERS
}

}  // namespace mcskin
