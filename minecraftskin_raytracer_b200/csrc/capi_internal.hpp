// capi_internal.hpp — what the units of the C ABI layer share (context.cu, frame.cu, host_out.cu, batch.cu, capi.cu):
// the context, its buffers and options, error reporting, and the functions one unit calls in another.
#pragma once
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "host_copy.hpp"
#include "host_prep.hpp"
#include "kernels.cuh"
#include "wavefront.cuh"
#include "mcskin_cuda.h"

using namespace mcskin;

inline int fail(int code, const std::string& msg) {
    set_last_error(msg);
    return code;
}
inline int cuda_fail(cudaError_t e, const char* what) {
    return fail(e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? MC_ERR_NO_DEVICE : MC_ERR_CUDA,
                std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU_TRY(expr)                                     \
    do {                                                 \
        cudaError_t e__ = (expr);                        \
        if (e__ != cudaSuccess) return cuda_fail(e__, #expr); \
    } while (0)

// Bumped whenever a device buffer is reallocated: captured frame graphs hold raw pointers.
extern std::atomic<unsigned long long> g_allocEpoch;

// A buffer that only ever grows, freed with its owner: device memory, or page-locked host memory.
template <bool kPinned>
struct GrowBuf {
    void* p = nullptr;
    size_t cap = 0;
    GrowBuf() = default;
    GrowBuf(const GrowBuf&) = delete;
    GrowBuf& operator=(const GrowBuf&) = delete;
    ~GrowBuf() { release(); }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (!kPinned) g_allocEpoch.fetch_add(1);
        release();
        cudaError_t e = kPinned ? cudaMallocHost(&p, bytes) : cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) (kPinned ? cudaFreeHost : cudaFree)(p);
        p = nullptr;
        cap = 0;
    }
};
using DevBuf = GrowBuf<false>;
using PinnedBuf = GrowBuf<true>;

struct PixelRect {
    int x, y, w, h;
};

// The options of a context (mcskin_cuda_context_set_option, INTEGRATION.md §6) with their defaults; kOptions describes them.
struct McOptions {
    int forceAllActive = 0;
    long long recordBudgetBytes = 1ll << 31;
    int shadeBlocksPerSm = 8;
    int softBlocksPerSm = 4;                 // persistent blocks of the soft-shadow kernel (its shared memory fits 4 per SM)
    int heavyTilesPerSm = 16;                // the figure's tiles are split over more blocks while a frame (all lanes) has fewer tiles per SM
    int primaryBlocksPerSm = 8;              // split tiles over blocks while a frame (all lanes) has fewer tiles than this per SM
                                             // (free of extra work: every block starts at its own round of the tile's stream)
    int waveQueuePct = 0;                    // hit-queue entries as a percentage of the paths (0: paths x (bounces + 1),
                                             // which cannot overflow; smaller queues redo overflowing paths in-thread)
    int frameLanes = 2;                      // a frame's tile rows are rendered on this many streams at once
    int cacheTileSeeds = 1;
    int overlapCopyOut = 2;                  // 0: copy after the frame; 1: whole image after the primary pass + the figure's
                                             // rectangle again at the end; 2: two destinations (see render_host)
    // The launches of a frame replayed as one CUDA graph (a frame is ~14 short kernels per lane;
    // launching them one by one costs the host more than the device needs to run them).  A graph
    // is captured the second time the same frame description is rendered and replayed while
    // nothing it depends on changes.
    int useGraphs = 1;
    int shadeMode = 0;                       // 0 wavefront, 1 megakernel (block groups), 2 megakernel (warp groups)
    long long waveBudgetBytes = 12ll << 30;  // queue storage; pixels beyond it fall back to the megakernel
    int shadowSeedMemo = 1;
    int stagedCopyOut = 1;                   // pageable destinations are filled piece by piece during the frame
    int batchLanes = 4;
    int batchGroup = 128;                    // scenes rendered by one set of launches (gridDim.y)
    int batchMode = 1;                       // 1: grouped launches, 0: one frame at a time over the lanes
    int debugPrimaryTiming = 0;              // the primary pass records when its blocks ran (blockTimes)
};
constexpr size_t kOptionCount = 19;  // the rows of kOptions

struct McContext : McOptions {
    int device = 0;
    int smCount = 148;
    cudaStream_t stream = nullptr;  // used when the caller passes stream 0 to the host-facing calls
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evCopy = nullptr;
    std::vector<cudaEvent_t> passEvents;  // 3 per chunk: before primary, between, after shade
    bool hasScene = false;
    PreparedFrame prep;
    DevBuf boxes, texels;
    DevBuf slotPixel, records;
    DevBuf imgF32, imgU8;
    DevBuf tileStates;           // seeded mt19937 state of every tile of a chunk
    DevBuf blockTimes;           // "debug_primary_timing": 4 words per block of the last primary launch
    int blockTimesCount = 0;
    DevBuf tileMap;              // render_tiles_into_frame: frame tile indices, heavy tiles first
    std::vector<int32_t> tileMapHost, tileMapOrdered;
    std::vector<PixelRect> tileMapLightRects;  // the tiles of the map the figure's rectangle does not touch, as rectangles
    unsigned long long tileMapVersion = 0;
    int tileMapHeavy = 0;
    DevFrame tileMapFrame{};     // the frame description the map was ordered for
    DevBuf wave;                 // queues of the wavefront shading pipeline
    PinnedBuf pinned;
    bool isChild = false;                    // a lane of another context (never splits frames itself)
    // seeded tile engines kept from the previous frame: they depend on the image width, the tile
    // size and the tile rows of the band only (tile_renderer.cpp:78), not on the scene
    struct TileSeedKey {
        int width = 0, tile_size = 0, first = 0, stride = 0, rows = 0;
        const void* buf = nullptr;
        cudaStream_t stream = nullptr;
        const void* map = nullptr;
        unsigned long long mapVersion = 0;
        int wordsPerPixel = 0, statesPerTile = 0;  // the per-round states of split tiles depend on the sampling pattern
        bool operator==(const TileSeedKey& o) const {
            return width == o.width && tile_size == o.tile_size && first == o.first && stride == o.stride &&
                   rows == o.rows && buf == o.buf && stream == o.stream && map == o.map && mapVersion == o.mapVersion &&
                   wordsPerPixel == o.wordsPerPixel && statesPerTile == o.statesPerTile;
        }
    } tileSeedKey;
    bool tileSeedValid = false;
    int splitLastRender = 0;                 // lanes (beyond this context) used by the last render
    cudaEvent_t evPrimaryDone = nullptr;     // (disable-timing) recorded after this lane's primary pass
    cudaStream_t copyStream = nullptr;       // device -> host copies that overlap the shading pass
    cudaEvent_t evFrameDone = nullptr;
    cudaEvent_t evUpload = nullptr;          // (disable-timing) recorded after the scene upload on ctx->stream
    unsigned long long seedGen = 0;          // bumped whenever tileStates is rewritten outside a graph
    bool capturing = false;                  // the launches are being captured into a graph: no timing events
    struct GraphKey {
        DevFrame frame;
        const void *blob, *texels, *outF32, *outU8;
        unsigned int blobBytes;
        int first, stride, lanes;
        const void* tileMap;
        unsigned long long mapVersion;
        int nTiles, nHeavy;
        const void *hotF32, *hotU8;
        const void *aovCoverage, *aovDepth, *aovTriId;  // a graph with AOV stores is never replayed without them, or vice versa
        const void *aovNormal, *aovAlbedo, *aovTexel;
        long long optionBits[kOptionCount];             // the launch options (0 for the others)
        unsigned long long allocEpoch;
        bool operator==(const GraphKey& o) const { return std::memcmp(this, &o, sizeof(GraphKey)) == 0; }
    };
    GraphKey graphKey{}, graphCandidate{};
    bool hasCandidate = false;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graphExec = nullptr;
    std::vector<unsigned long long> graphSeedGens;  // seedGen of every lane when the graph was captured
    std::vector<int> graphLaneLaunches, graphLaneChunks, graphLaneTiles;
    bool graphLastRender = false;
    // stats of the last render
    McRenderStats stats{};
    bool statsPending = false;
    bool uploadQueued = false;             // evUpload has been recorded at least once
    DevBuf countLog;                       // one counter per chunk of the last render
    PinnedBuf countHost;                   // ... and where the frame's last kernel (or a copy) leaves them for the statistics
    unsigned int* countAlias = nullptr;    // countHost as the device addresses it (null: not mapped)
    PinnedBuf sceneStage;                  // page-locked staging of the scene blob and texels (upload_scene)
    DevBuf seedMemo;                       // FreshStream::seed_memo's table (dev_mt19937.cuh), shared with the lanes
    PinnedBuf stageF32, stageU8;           // page-locked staging images for pageable destinations (render_host_staged)
    std::vector<cudaEvent_t> pieceEvents;  // one per piece of the staging image on its way to the host
    std::vector<std::pair<const void*, bool>> farCache;  // is_far_memory
    int chunksLastRender = 0;
    // batch rendering
    DevBuf batchScenes, batchSlots, batchRecords, batchWave, batchCounts;
    DevBuf batchSkinSrc;                     // render_skin_batch: per skin the raw atlas, its face table, the slicing job
    PinnedBuf batchSkinStage[2];
    std::vector<McBox> batchSkinBoxes;
    PinnedBuf batchStage[2];
    cudaEvent_t evStage[2] = {nullptr, nullptr};
    std::vector<PreparedFrame> batchPreps;
    std::vector<McContext*> lanes;
    // AOV planes the render calls write next to the colour (mcskin_cuda_context_set_aov_targets; device-addressable
    // pointers, all null: none).  Child lanes get their parent's (inherit_options).
    McAovTargets aov{};
    DevBuf aovPlanes;                        // mcskin_cuda_render_aovs: the planes on the device before they go to the host
    DevBuf pngScratch;                       // mcskin_cuda_context_encode_png: filtered streams, tokens, segments (png.cuh)
};

// The launchers of one of the three builds of the hot kernels (dev_types.cuh): the general form; no pose code, for
// scenes in which no box is posed; counter-based random streams.
struct KernelBuild {
    decltype(&mcskin::launch_primary) launch_primary;
    decltype(&mcskin::launch_shade) launch_shade;
    decltype(&mcskin::launch_wavefront) launch_wavefront;
    decltype(&mcskin::launch_primary_batch) launch_primary_batch;
};
constexpr KernelBuild kGeneralBuild{&launch_primary, &launch_shade, &launch_wavefront, &launch_primary_batch};
constexpr KernelBuild kPlainBuild{&plain::launch_primary, &plain::launch_shade, &plain::launch_wavefront, &plain::launch_primary_batch};
constexpr KernelBuild kCounterBuild{&counter::launch_primary, &counter::launch_shade, &counter::launch_wavefront,
                                    &counter::launch_primary_batch};

inline const KernelBuild& kernels_for(const DevFrame& f) { return f.rng_mode ? kCounterBuild : (f.any_rotated ? kGeneralBuild : kPlainBuild); }

inline bool aov_on(const McContext* ctx) { return aov_any(&ctx->aov); }
// the planes of the image that starts `pixels` pixels into the targets (image i of a batch)
inline McAovTargets aov_at(const McAovTargets& a, size_t pixels) {
    McAovTargets r{};
    r.coverage = a.coverage ? a.coverage + pixels : nullptr;
    r.depth = a.depth ? a.depth + pixels : nullptr;
    r.tri_id = a.tri_id ? a.tri_id + pixels : nullptr;
    r.normal = a.normal ? a.normal + 3 * pixels : nullptr;
    r.albedo = a.albedo ? a.albedo + 4 * pixels : nullptr;
    r.texel = a.texel ? a.texel + pixels : nullptr;
    return r;
}

// What one launch sequence covers: tile rows {first + k*stride} written at tile rows outFirst + k*outStride of
// the output image, or (map != null) any set of whole tiles — a device array of frame tile indices, the
// nHeavy tiles that intersect the figure's screen rectangle first — written at their own place in a full frame.
struct BandSpec {
    int first = 0, stride = 1, outFirst = 0, outStride = 1;
    const int* map = nullptr;
    int nTiles = 0, nHeavy = 0;
    unsigned long long mapVersion = 0;
    float4* hotF32 = nullptr;  // BandView::hot_*: where the tiles the figure's rectangle touches are written instead
    uchar4* hotU8 = nullptr;
};

// The context's device image(s) of `pixels` pixels for the outputs that are wanted (null for the others).
struct DeviceImage {
    float4* f32;
    uchar4* u8;
};
inline int device_image(McContext* ctx, bool wantF32, bool wantU8, size_t pixels, DeviceImage* out) {
    if (wantF32) CU_TRY(ctx->imgF32.reserve(pixels * sizeof(float4)));
    if (wantU8) CU_TRY(ctx->imgU8.reserve(pixels * sizeof(uchar4)));
    out->f32 = wantF32 ? static_cast<float4*>(ctx->imgF32.p) : nullptr;
    out->u8 = wantU8 ? static_cast<uchar4*>(ctx->imgU8.p) : nullptr;
    return MC_OK;
}

// context.cu
extern std::mutex g_ctxMutex;  // held by the host-facing calls that use the per-device shared contexts
int shared_context(int device, McContext** out);
int upload_scene(McContext* ctx);
int finish_stats(McContext* ctx, McRenderStats* out);
void inherit_options(McContext* lane, const McContext* ctx);
void launch_option_bits(const McContext* ctx, long long* bits);

// frame.cu
FramePointers frame_pointers(const McContext* ctx);
uint2* seed_memo_of(McContext* ctx);
int ensure_lanes(McContext* ctx, int n);
int render_bands(McContext* ctx, int first, int stride, float4* outF32, uchar4* outU8, cudaStream_t stream,
                 bool frameLayout = false, const BandSpec* tiles = nullptr, float4* hotF32 = nullptr, uchar4* hotU8 = nullptr);
std::vector<PixelRect> tile_rects(const DevFrame& f, std::vector<int32_t> tiles);
int prepare_tile_map(McContext* ctx, const int32_t* tiles, int32_t nTiles, cudaStream_t s, BandSpec* spec, bool* empty);
