// capi.cu — the extern "C" layer of include/mcskin_cuda.h: contexts, device memory,
// launches, host<->device copies.  No exceptions leave this file; every failure is a
// negative MC_ERR_* plus a thread-local message (mcskin_cuda_last_error).
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

namespace {

int fail(int code, const std::string& msg) {
    set_last_error(msg);
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    return fail(e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? MC_ERR_NO_DEVICE : MC_ERR_CUDA,
                std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU_TRY(expr)                                     \
    do {                                                 \
        cudaError_t e__ = (expr);                        \
        if (e__ != cudaSuccess) return cuda_fail(e__, #expr); \
    } while (0)

// Bumped whenever a device buffer is reallocated: captured frame graphs hold raw pointers.
std::atomic<unsigned long long> g_allocEpoch{1};

// Device buffer that only ever grows.
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        g_allocEpoch.fetch_add(1);
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};
struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMallocHost(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

struct PixelRect {
    int x, y, w, h;
};

}  // namespace

struct McContext {
    int device = 0;
    int smCount = 148;
    cudaStream_t stream = nullptr;  // used when the caller passes stream 0 to the host-facing calls
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evCopy = nullptr;
    std::vector<cudaEvent_t> passEvents;  // 3 per chunk: before primary, between, after shade
    bool hasScene = false;
    PreparedFrame prep;
    McConfig cfg{};
    DevBuf boxes, texels;
    DevBuf count, slotPixel, records;
    DevBuf imgF32, imgU8, scratchIn, scratchOut;
    DevBuf tileStates;           // seeded mt19937 state of every tile of a chunk
    DevBuf blockTimes;           // "debug_primary_timing": 4 words per block of the last primary launch
    int debugPrimaryTiming = 0;
    int blockTimesCount = 0;
    DevBuf tileMap;              // render_tiles_into_frame: frame tile indices, heavy tiles first
    std::vector<int32_t> tileMapHost, tileMapOrdered;
    std::vector<PixelRect> tileMapLightRects;  // the tiles of the map the figure's rectangle does not touch, as rectangles
    unsigned long long tileMapVersion = 0;
    int tileMapHeavy = 0;
    DevFrame tileMapFrame{};     // the frame description the map was ordered for
    DevBuf wave;                 // queues of the wavefront shading pipeline
    PinnedBuf pinned;
    // options
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
    int cacheTileSeeds = 1;
    int splitLastRender = 0;                 // lanes (beyond this context) used by the last render
    cudaEvent_t evPrimaryDone = nullptr;     // (disable-timing) recorded after this lane's primary pass
    cudaStream_t copyStream = nullptr;       // device -> host copies that overlap the shading pass
    cudaEvent_t evFrameDone = nullptr;
    int overlapCopyOut = 2;                  // 0: copy after the frame; 1: whole image after the primary pass + the figure's
                                             // rectangle again at the end; 2: two destinations (see render_host)
    cudaEvent_t evUpload = nullptr;          // (disable-timing) recorded after the scene upload on ctx->stream
    unsigned long long seedGen = 0;          // bumped whenever tileStates is rewritten outside a graph
    bool capturing = false;                  // the launches are being captured into a graph: no timing events
    // The launches of a frame replayed as one CUDA graph (a frame is ~14 short kernels per lane;
    // launching them one by one costs the host more than the device needs to run them).  A graph
    // is captured the second time the same frame description is rendered and replayed while
    // nothing it depends on changes.
    int useGraphs = 1;
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
        long long optionBits[12];
        unsigned long long allocEpoch;
        bool operator==(const GraphKey& o) const { return std::memcmp(this, &o, sizeof(GraphKey)) == 0; }
    };
    GraphKey graphKey{}, graphCandidate{};
    bool hasCandidate = false;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graphExec = nullptr;
    std::vector<unsigned long long> graphSeedGens;  // seedGen of every lane when the graph was captured
    int graphLaunches = 0, graphChunks = 0, graphSplit = 0;
    std::vector<int> graphLaneLaunches, graphLaneChunks, graphLaneTiles;
    bool graphLastRender = false;
    int shadeMode = 0;                       // 0 wavefront, 1 megakernel (block groups), 2 megakernel (warp groups)
    long long waveBudgetBytes = 12ll << 30;   // queue storage; pixels beyond it fall back to the megakernel
    // stats of the last render
    McRenderStats stats{};
    bool statsPending = false;
    bool uploadQueued = false;             // evUpload has been recorded at least once
    DevBuf countLog;                       // one counter per chunk of the last render
    PinnedBuf countHost;                   // ... and where the frame's last kernel (or a copy) leaves them for the statistics
    unsigned int* countAlias = nullptr;    // countHost as the device addresses it (null: not mapped)
    PinnedBuf sceneStage;                  // page-locked staging of the scene blob and texels (upload_scene)
    DevBuf seedMemo;                       // FreshStream::seed_memo's table (dev_mt19937.cuh), shared with the lanes
    int shadowSeedMemo = 1;                // option "shadow_seed_memo"
    PinnedBuf stageF32, stageU8;           // page-locked staging images for pageable destinations (render_host_staged)
    std::vector<cudaEvent_t> pieceEvents;  // one per piece of the staging image on its way to the host
    int stagedCopyOut = 1;                 // option "staged_copy_out": pageable destinations are filled piece by piece during the frame
    std::vector<std::pair<const void*, bool>> farCache;  // is_far_memory
    int chunksLastRender = 0;
    // batch rendering
    int batchLanes = 4;
    int batchGroup = 128;                    // scenes rendered by one set of launches (gridDim.y)
    int batchMode = 1;                       // 1: grouped launches, 0: one frame at a time over the lanes
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
};

namespace {

bool aov_on(const McContext* ctx) { return ctx->aov.coverage || ctx->aov.depth || ctx->aov.tri_id; }
// the planes of the image that starts `pixels` pixels into the targets (image i of a batch)
McAovTargets aov_at(const McAovTargets& a, size_t pixels) {
    McAovTargets r{};
    r.coverage = a.coverage ? a.coverage + pixels : nullptr;
    r.depth = a.depth ? a.depth + pixels : nullptr;
    r.tri_id = a.tri_id ? a.tri_id + pixels : nullptr;
    return r;
}

int upload_scene(McContext* ctx) {
    const PreparedFrame& pf = ctx->prep;
    if (pf.blob.size() > kMaxSceneSmemBytes)
        return fail(MC_ERR_LIMIT, "scene has too many meshes for the shared-memory staging area (" +
                                      std::to_string(pf.boxes.size()) + " boxes)");
    CU_TRY(ctx->boxes.reserve(pf.blob.size()));
    CU_TRY(ctx->texels.reserve(pf.texels.size() * sizeof(float4h)));
    // Through a page-locked staging buffer: two host memcpys (~55 KB) and two copies the runtime only has to queue
    // (from pageable memory it stages them itself, synchronously: ~30 us per scene).  The host vectors may change
    // afterwards; the staging buffer is reused once the previous upload has left it; renders on another stream wait
    // for the event.
    const size_t blobBytes = (pf.blob.size() + 255) & ~size_t(255), texelBytes = pf.texels.size() * sizeof(float4h);
    if (ctx->uploadQueued) CU_TRY(cudaEventSynchronize(ctx->evUpload));
    CU_TRY(ctx->sceneStage.reserve(blobBytes + texelBytes + 256));
    unsigned char* stage = static_cast<unsigned char*>(ctx->sceneStage.p);
    std::memcpy(stage, pf.blob.data(), pf.blob.size());
    if (texelBytes) std::memcpy(stage + blobBytes, pf.texels.data(), texelBytes);
    CU_TRY(cudaMemcpyAsync(ctx->boxes.p, stage, pf.blob.size(), cudaMemcpyHostToDevice, ctx->stream));
    if (texelBytes) CU_TRY(cudaMemcpyAsync(ctx->texels.p, stage + blobBytes, texelBytes, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(cudaEventRecord(ctx->evUpload, ctx->stream));
    ctx->uploadQueued = true;
    return MC_OK;
}

FramePointers frame_pointers(const McContext* ctx) {
    return FramePointers{static_cast<const unsigned char*>(ctx->boxes.p), static_cast<const float4*>(ctx->texels.p),
                         static_cast<unsigned int>(ctx->prep.blob.size())};
}

int local_tile_rows(const DevFrame& f, int first, int stride) {
    if (f.tiles_y <= 0 || first < 0 || stride <= 0 || first >= f.tiles_y) return 0;
    return (f.tiles_y - first + stride - 1) / stride;
}

int band_pixel_rows(const DevFrame& f, int first, int stride) {
    const int n = local_tile_rows(f, first, stride);
    if (n == 0) return 0;
    const int lastTileRow = first + (n - 1) * stride;
    const int lastHeight = std::min(f.tile_size, f.height - lastTileRow * f.tile_size);
    return (n - 1) * f.tile_size + lastHeight;
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

// The table of FreshStream::seed_memo, allocated and zeroed the first time a frame with soft shadows comes in (never
// inside a graph capture: the frame that is captured has been rendered once before).  Null when switched off.
static uint2* seed_memo_of(McContext* ctx) {
    if (!ctx->shadowSeedMemo) return nullptr;
    if (!ctx->seedMemo.p) {
        if (ctx->capturing) return nullptr;
        const size_t bytes = static_cast<size_t>(kSeedMemoEntries) * sizeof(uint2);
        if (ctx->seedMemo.reserve(bytes) != cudaSuccess || cudaMemsetAsync(ctx->seedMemo.p, 0, bytes, ctx->stream) != cudaSuccess ||
            cudaStreamSynchronize(ctx->stream) != cudaSuccess) {  // (zeroed before any stream of a frame can read it)
            cudaGetLastError();
            ctx->seedMemo.release();
            ctx->shadowSeedMemo = 0;  // no memory for it: the frames are the same without
            return nullptr;
        }
    }
    return static_cast<uint2*>(ctx->seedMemo.p);
}

// Is p (an output image the kernels store to) anything but this context's device memory: a mapped host range, a
// peer device's allocation?  The last answers are kept: the pointers of a render loop repeat.
static bool is_far_memory(McContext* ctx, const void* p) {
    if (!p) return false;
    for (const auto& e : ctx->farCache)
        if (e.first == p) return e.second;
    cudaPointerAttributes attr{};
    bool far = false;
    if (cudaPointerGetAttributes(&attr, p) == cudaSuccess) far = attr.type == cudaMemoryTypeHost || (attr.type == cudaMemoryTypeDevice && attr.device != ctx->device);
    else cudaGetLastError();
    if (ctx->farCache.size() >= 8) ctx->farCache.erase(ctx->farCache.begin());
    ctx->farCache.emplace_back(p, far);
    return far;
}

// Launches the two passes of a band on one stream; output pointers are device memory.  scn: the context whose
// scene (prepared frame, box and texel buffers) is rendered.
int render_bands_lane(McContext* ctx, const McContext* scn, const BandSpec& spec, float4* outF32, uchar4* outU8,
                      cudaStream_t stream, int lanesInFlight = 1) {
    const DevFrame& f = scn->prep.frame;
    const bool mapped = spec.map != nullptr;
    const int first = spec.first, stride = spec.stride;
    const int nRows = mapped ? 0 : local_tile_rows(f, first, stride);
    const long long nTilesAll = mapped ? spec.nTiles : static_cast<long long>(nRows) * f.tiles_x;
    ctx->chunksLastRender = 0;
    ctx->graphLastRender = false;
    ctx->stats = McRenderStats{};
    ctx->stats.n_samples = static_cast<int64_t>(std::max(f.width, 0)) * std::max(f.height, 0) * f.spp;
    ctx->stats.n_tiles = nTilesAll;
    if (nTilesAll == 0) return MC_OK;
    if (f.width > 65535 || f.height > 65535) return fail(MC_ERR_LIMIT, "image larger than 65535 pixels on a side");
    if (static_cast<long long>(f.tile_size) * f.tile_size > (1ll << 30))
        return fail(MC_ERR_LIMIT, "tile_size too large");

    const bool classify = !ctx->forceAllActive && f.spp <= kBlockThreads;
    // A band is rendered in chunks of UNITS — whole tile rows, or tiles of the map — so that the worst-case
    // work list of a chunk fits the budget.  Work-list slots a unit can need: every pixel, or, as the
    // classifying primary pass only lists pixels inside the figure's screen rectangle, the rectangle's columns
    // of a tile row / the pixels of a tile that intersects it (the first nHeavy of a map).
    const size_t tilePixels = static_cast<size_t>(f.tile_size) * f.tile_size;
    size_t slotsPerUnit = mapped ? tilePixels : static_cast<size_t>(f.tiles_x) * tilePixels;
    if (!mapped && classify && f.rect_valid) {
        const long long rectW = static_cast<long long>(std::min(f.width - 1, f.rect_x1)) - std::max(0, f.rect_x0) + 1;
        slotsPerUnit = std::min(slotsPerUnit, static_cast<size_t>(std::max<long long>(rectW, 1)) * f.tile_size);
    }
    const size_t nUnits = mapped ? static_cast<size_t>(spec.nTiles) : static_cast<size_t>(nRows);
    const size_t tilesPerUnit = mapped ? 1 : static_cast<size_t>(f.tiles_x);
    // units that can list pixels at all (the rest need no slots): every row; the heavy tiles of a map
    const size_t nListingUnits = (mapped && classify && f.rect_valid) ? static_cast<size_t>(spec.nHeavy) : nUnits;
    const size_t recordBytesPerSlot = static_cast<size_t>(f.spp) * f.draws_per_sample * sizeof(float);
    size_t unitsPerChunk = nUnits;
    if (recordBytesPerSlot > 0 && nListingUnits > 0) {
        const size_t perUnit = slotsPerUnit * recordBytesPerSlot;
        const size_t fit = std::max<size_t>(1, static_cast<size_t>(ctx->recordBudgetBytes) / std::max<size_t>(1, perUnit));
        // (a map lists its heavy tiles first: chunks of `fit` units hold at most `fit` listing units each)
        if (fit < nListingUnits) unitsPerChunk = fit;
    }
    // slot indices are 32-bit
    while (unitsPerChunk > 1 && std::min(unitsPerChunk, nListingUnits) * slotsPerUnit > 0x7fffffffull) --unitsPerChunk;
    const size_t slotCap = std::max<size_t>(1, std::min(unitsPerChunk, std::max<size_t>(nListingUnits, 0)) * slotsPerUnit);
    if (slotCap > 0x7fffffffull) return fail(MC_ERR_LIMIT, "one tile row holds more than 2^31 pixels");
    const int nChunks = static_cast<int>((nUnits + unitsPerChunk - 1) / unitsPerChunk);

    CU_TRY(ctx->countLog.reserve(sizeof(unsigned int) * 2 * nChunks));  // [active count | group counter] per chunk
    if (ctx->countHost.cap < sizeof(unsigned int) * nChunks) {
        g_allocEpoch.fetch_add(1);  // (captured graphs copy to the old address)
        CU_TRY(ctx->countHost.reserve(sizeof(unsigned int) * std::max(1024, 2 * nChunks)));
        void* alias = nullptr;
        if (cudaHostGetDevicePointer(&alias, ctx->countHost.p, 0) != cudaSuccess) {
            cudaGetLastError();
            alias = nullptr;
        }
        ctx->countAlias = static_cast<unsigned int*>(alias);
    }
    unsigned int* const countAlias = ctx->countAlias;
    CU_TRY(ctx->slotPixel.reserve(slotCap * sizeof(uint2)));
    CU_TRY(ctx->records.reserve(std::max<size_t>(16, slotCap * recordBytesPerSlot)));
    // Splitting the figure's tiles pays only when the frame (all lanes in flight) has too few tiles to
    // keep every SM busy for as long as its slowest tile takes: below ~10 tiles per SM (B200 sweep:
    // a whole 1080p frame, 2040 tiles, is best unsplit; half a frame is best split in three).
    const long long tilesInFlight = nTilesAll * std::max(1, lanesInFlight);
    const int heavyTarget = tilesInFlight * 3 >= 2ll * ctx->smCount * ctx->heavyTilesPerSm
                                ? 0 : ctx->smCount * ctx->heavyTilesPerSm / std::max(1, lanesInFlight);
    const int primaryTarget = ctx->smCount * ctx->primaryBlocksPerSm / std::max(1, lanesInFlight);
    // engine states per tile: one per round of 256 pixels when tiles are split over blocks (kernels.cu)
    const size_t statesPerTile = static_cast<size_t>(primary_states_per_tile(
        f, static_cast<int>(std::min<size_t>(unitsPerChunk * tilesPerUnit, 0x7fffffff)), 1, primaryTarget, heavyTarget));
    CU_TRY(ctx->tileStates.reserve(std::max<size_t>(16, unitsPerChunk * tilesPerUnit * statesPerTile * 624 * sizeof(uint32_t))));
    CU_TRY(cudaMemsetAsync(ctx->countLog.p, 0, sizeof(unsigned int) * 2 * nChunks, stream));

    while (ctx->passEvents.size() < static_cast<size_t>(3 * nChunks)) {
        cudaEvent_t e;
        CU_TRY(cudaEventCreate(&e));
        ctx->passEvents.push_back(e);
    }
    // wavefront storage: per path (terminal colour, bounce stack) and per hit-queue entry.  A queue of
    // paths x (bounces + 1) entries cannot overflow; if the budget does not allow it the queue shrinks (to no
    // less than 1.25 entries per path; paths whose hits do not fit are redone in-thread), then the number of
    // paths does (pixels beyond them are shaded by the megakernel).
    WaveView wave{};
    const bool aov = aov_on(ctx);
    AovView aovView{};
    aovView.planes = ctx->aov;
    if (ctx->shadeMode == 0) {
        const size_t perPath = wavefront_bytes_per_path(f, aov), perEntry = wavefront_bytes_per_entry();
        const size_t hitsMax = static_cast<size_t>(wavefront_max_hits_per_path(f));
        const size_t budget = static_cast<size_t>(ctx->waveBudgetBytes);
        const size_t worstPaths = slotCap * static_cast<size_t>(f.spp);
        size_t paths = std::min(worstPaths, budget / (perPath + perEntry * std::min<size_t>(hitsMax, 2)));
        paths = std::min<size_t>(paths, 0x7fffff00u);
        paths = std::max<size_t>(paths, static_cast<size_t>(f.spp));
        size_t entries = paths * hitsMax;
        if (ctx->waveQueuePct > 0) entries = std::min(entries, std::max<size_t>(32, paths * static_cast<size_t>(ctx->waveQueuePct) / 100));
        const size_t room = budget > paths * perPath ? (budget - paths * perPath) / perEntry : 0;
        entries = std::min(entries, std::max(room, paths + paths / 4));
        entries = std::min<size_t>(entries, 0xffffff00u);
        const size_t bytes = paths * perPath + entries * perEntry + wavefront_fixed_bytes(f) + 16 * 256;
        CU_TRY(ctx->wave.reserve(bytes));
        if (!wavefront_carve(f, ctx->wave.p, ctx->wave.cap, static_cast<unsigned int>(paths), static_cast<unsigned int>(entries),
                             ctx->smCount * ctx->shadeBlocksPerSm, &wave, aov ? &aovView : nullptr))
            return fail(MC_ERR_CUDA, "wavefront buffer carve failed");
        wave.softGrid = ctx->smCount * ctx->softBlocksPerSm;
        wave.seedMemo = static_cast<uint2*>(scn->seedMemo.p);  // (render_bands has seen to it; the lanes of a frame share it)
        if (!scn->shadowSeedMemo) wave.seedMemo = nullptr;
    }
    if (!ctx->capturing) CU_TRY(cudaEventRecord(ctx->ev0, stream));
    const FramePointers fp = frame_pointers(scn);
    int launches = 0;
    McContext::TileSeedKey seedKey;
    seedKey.width = f.width; seedKey.tile_size = f.tile_size; seedKey.first = first; seedKey.stride = stride;
    seedKey.rows = mapped ? spec.nTiles : nRows; seedKey.buf = ctx->tileStates.p; seedKey.stream = stream;
    seedKey.map = spec.map; seedKey.mapVersion = spec.mapVersion;
    seedKey.wordsPerPixel = f.spp * f.draws_per_sample; seedKey.statesPerTile = static_cast<int>(statesPerTile) | (f.rng_mode << 16);
    const bool seedsCacheable = ctx->cacheTileSeeds && nChunks == 1 && f.draws_per_sample > 0;
    const bool seedTiles = !(seedsCacheable && ctx->tileSeedValid && seedKey == ctx->tileSeedKey);
    ctx->tileSeedKey = seedKey;
    ctx->tileSeedValid = false;
    if (seedTiles) ++ctx->seedGen;
    // where the shaded pixels go: this device's memory, or across a link (BandView::far_output)
    const bool farOutput = spec.hotF32 || spec.hotU8 || is_far_memory(ctx, outF32) || is_far_memory(ctx, outU8);
    for (int c = 0; c < nChunks; ++c) {
        const size_t unit0 = static_cast<size_t>(c) * unitsPerChunk;
        const size_t units = std::min<size_t>(unitsPerChunk, nUnits - unit0);
        BandView band{};
        band.out_f32 = outF32;
        band.out_u8 = outU8;
        band.hot_f32 = spec.hotF32;
        band.hot_u8 = spec.hotU8;
        band.far_output = farOutput ? 1 : 0;
        if (ctx->debugPrimaryTiming && nChunks == 1) {  // room for the finest split: one block per 256-pixel round of every tile
            const size_t blocks = static_cast<size_t>(nTilesAll) * ((tilePixels + kBlockThreads - 1) / kBlockThreads);
            CU_TRY(ctx->blockTimes.reserve(blocks * 4 * sizeof(unsigned long long)));
            CU_TRY(cudaMemsetAsync(ctx->blockTimes.p, 0, blocks * 4 * sizeof(unsigned long long), stream));
            band.block_times = static_cast<unsigned long long*>(ctx->blockTimes.p);
            ctx->blockTimesCount = static_cast<int>(blocks);
        }
        size_t listing = units;
        if (mapped) {
            band.tile_map = spec.map + unit0;
            band.n_tiles = static_cast<int>(units);
            band.n_heavy = static_cast<int>(unit0 >= static_cast<size_t>(spec.nHeavy) ? 0 : std::min<size_t>(units, spec.nHeavy - unit0));
            if (classify && f.rect_valid) listing = static_cast<size_t>(band.n_heavy);
        } else {
            band.first_tile_row = first + static_cast<int>(unit0) * stride;
            band.tile_row_stride = stride;
            band.n_tile_rows = static_cast<int>(units);
            band.out_first_row = spec.outFirst + static_cast<int>(unit0) * spec.outStride;
            band.out_row_stride = spec.outStride;
        }
        ActiveList list;
        list.count = static_cast<unsigned int*>(ctx->countLog.p) + c;
        list.slot_pixel = static_cast<uint2*>(ctx->slotPixel.p);
        list.records = static_cast<float*>(ctx->records.p);
        list.capacity = static_cast<unsigned int>(std::min(slotCap, std::max<size_t>(1, listing * slotsPerUnit)));
        // the wavefront's last kernel leaves the count in page-locked host memory for the statistics (no copy, nothing
        // more in the stream); the other shading modes copy it below
        list.count_host = (ctx->shadeMode == 0 && countAlias) ? countAlias + c : nullptr;
        if (!classify) {
            // positional slots: mark all unused, preset the count to the capacity
            CU_TRY(cudaMemsetAsync(list.slot_pixel, 0xff, static_cast<size_t>(list.capacity) * sizeof(uint2), stream));
            CU_TRY(cudaMemcpyAsync(list.count, &list.capacity, sizeof(unsigned int), cudaMemcpyHostToDevice, stream));
        }
        if (!ctx->capturing) CU_TRY(cudaEventRecord(ctx->passEvents[3 * c], stream));
        if (aov) {  // every pixel of the chunk gets the defaults; the shading pass overwrites the ones it resolves
            launch_aov_defaults(f, band, ctx->aov, nullptr, 1, stream);
            ++launches;
        }
        // (three builds of the kernels — dev_types.cuh: counter-based random streams; no pose code, for scenes in which
        // no box is posed; the general form)
        const int build = f.rng_mode ? 2 : (f.any_rotated ? 0 : 1);
        uint32_t* const states = static_cast<uint32_t*>(ctx->tileStates.p);
        const bool seeded =
            build == 2 ? counter::launch_primary(f, fp, band, list, classify ? 1 : 0, states, seedTiles, primaryTarget, heavyTarget, stream)
            : build == 1 ? plain::launch_primary(f, fp, band, list, classify ? 1 : 0, states, seedTiles, primaryTarget, heavyTarget, stream)
                         : launch_primary(f, fp, band, list, classify ? 1 : 0, states, seedTiles, primaryTarget, heavyTarget, stream);
        ctx->tileSeedValid = seedsCacheable && seeded;
        // from here on every pixel of the band outside the figure's screen rectangle is final: the host
        // copy of the image may start (render_host).  Inside a capture this must be a real event-record
        // node, visible to streams outside the graph.
        if (c == nChunks - 1)
            CU_TRY(cudaEventRecordWithFlags(ctx->evPrimaryDone, stream, ctx->capturing ? cudaEventRecordExternal : cudaEventRecordDefault));
        if (!ctx->capturing) CU_TRY(cudaEventRecord(ctx->passEvents[3 * c + 1], stream));
        unsigned int* groupCounter = static_cast<unsigned int*>(ctx->countLog.p) + nChunks + c;
        const int shadeGrid = ctx->smCount * ctx->shadeBlocksPerSm;
        if (ctx->shadeMode == 0) {
            if (build == 2) counter::launch_wavefront(f, fp, band, list, wave, groupCounter, stream, &launches, nullptr, 1, aov ? &aovView : nullptr);
            else if (build == 1) plain::launch_wavefront(f, fp, band, list, wave, groupCounter, stream, &launches, nullptr, 1, aov ? &aovView : nullptr);
            else launch_wavefront(f, fp, band, list, wave, groupCounter, stream, &launches, nullptr, 1, aov ? &aovView : nullptr);
        } else {
            if (build == 2) launches += counter::launch_shade(f, fp, band, list, shadeGrid, groupCounter, 0u, stream, ctx->shadeMode, &ctx->aov);
            else if (build == 1) launches += plain::launch_shade(f, fp, band, list, shadeGrid, groupCounter, 0u, stream, ctx->shadeMode, &ctx->aov);
            else launches += launch_shade(f, fp, band, list, shadeGrid, groupCounter, 0u, stream, ctx->shadeMode, &ctx->aov);
        }
        if (!ctx->capturing) CU_TRY(cudaEventRecord(ctx->passEvents[3 * c + 2], stream));
        ++launches;
    }
    if (!(ctx->shadeMode == 0 && countAlias))
        CU_TRY(cudaMemcpyAsync(ctx->countHost.p, ctx->countLog.p, sizeof(unsigned int) * nChunks, cudaMemcpyDeviceToHost, stream));
    if (!ctx->capturing) CU_TRY(cudaEventRecord(ctx->ev1, stream));
    CU_TRY(cudaGetLastError());
    ctx->chunksLastRender = nChunks;
    ctx->stats.n_kernel_launches = launches;
    ctx->statsPending = true;
    return MC_OK;
}

int ensure_lanes(McContext* ctx, int n) {
    while (static_cast<int>(ctx->lanes.size()) < n) {
        McContext* lane = nullptr;
        const int rc = mcskin_cuda_context_create(ctx->device, &lane);
        if (rc != MC_OK) return rc;
        lane->isChild = true;
        ctx->lanes.push_back(lane);
    }
    return MC_OK;
}

void inherit_options(McContext* lane, const McContext* ctx) {
    lane->shadeMode = ctx->shadeMode;
    lane->forceAllActive = ctx->forceAllActive;
    lane->waveQueuePct = ctx->waveQueuePct;
    lane->waveBudgetBytes = ctx->waveBudgetBytes;
    lane->recordBudgetBytes = ctx->recordBudgetBytes;
    lane->shadeBlocksPerSm = ctx->shadeBlocksPerSm;
    lane->softBlocksPerSm = ctx->softBlocksPerSm;
    lane->primaryBlocksPerSm = ctx->primaryBlocksPerSm;
    lane->heavyTilesPerSm = ctx->heavyTilesPerSm;
    lane->cacheTileSeeds = ctx->cacheTileSeeds;
    lane->aov = ctx->aov;
    lane->useGraphs = 0;
}

// Launches the lanes of one frame (see render_bands) on `stream` and the child lanes' streams.
// frameLayout: the output is a full-frame image and every tile row lands at its own frame position
// (output tile row = frame tile row) instead of a compact band.
int launch_frame_lanes(McContext* ctx, int first, int stride, int L, float4* outF32, uchar4* outU8, cudaStream_t stream,
                       bool frameLayout, const BandSpec* tiles, float4* hotF32, uchar4* hotU8) {
    if (tiles) {  // a tile map is one lane
        BandSpec t = *tiles;
        t.hotF32 = hotF32; t.hotU8 = hotU8;
        return render_bands_lane(ctx, ctx, t, outF32, outU8, stream);
    }
    auto rows = [&](int f0, int st, int out0, int outSt) {
        BandSpec b;
        b.first = f0; b.stride = st; b.outFirst = out0; b.outStride = outSt;
        b.hotF32 = hotF32; b.hotU8 = hotU8;
        return b;
    };
    if (L <= 1)
        return render_bands_lane(ctx, ctx, rows(first, stride, frameLayout ? first : 0, frameLayout ? stride : 1), outF32, outU8, stream);
    CU_TRY(cudaEventRecord(ctx->evCopy, stream));  // fork point
    // lane 0 on the caller's stream, lanes 1..L-1 on their own
    int rc = render_bands_lane(ctx, ctx, rows(first, stride * L, frameLayout ? first : 0, frameLayout ? stride * L : L), outF32, outU8, stream, L);
    if (rc != MC_OK) return rc;
    for (int k = 1; k < L; ++k) {
        McContext* lane = ctx->lanes[k - 1];
        CU_TRY(cudaStreamWaitEvent(lane->stream, ctx->evCopy, 0));
        rc = render_bands_lane(lane, ctx, rows(first + k * stride, stride * L, frameLayout ? first + k * stride : k,
                                               frameLayout ? stride * L : L), outF32, outU8, lane->stream, L);
        if (rc != MC_OK) return rc;
        CU_TRY(cudaEventRecord(lane->evCopy, lane->stream));
    }
    for (int k = 1; k < L; ++k) CU_TRY(cudaStreamWaitEvent(stream, ctx->lanes[k - 1]->evCopy, 0));  // join
    return MC_OK;
}

long long option_bits(const McContext* c, int i) {
    const long long v[12] = {c->forceAllActive, c->recordBudgetBytes, c->shadeBlocksPerSm, c->primaryBlocksPerSm,
                             c->waveQueuePct, c->shadeMode, c->waveBudgetBytes, c->shadowSeedMemo,
                             c->softBlocksPerSm, c->cacheTileSeeds, c->heavyTilesPerSm, c->frameLanes};
    return v[i];
}

void drop_graph(McContext* ctx) {
    if (ctx->graphExec) cudaGraphExecDestroy(ctx->graphExec);
    if (ctx->graph) cudaGraphDestroy(ctx->graph);
    ctx->graphExec = nullptr;
    ctx->graph = nullptr;
}

// Renders the tile rows {first + k*stride} of the context's scene into a compact band image.
// With frameLanes = L > 1 the rows are dealt round-robin to L streams (this context's and L-1
// child lanes with their own work lists and queues): the kernels of one lane are short and
// latency-bound towards the end of a frame (deep bounce levels, the tails of every launch), and
// the SMs fill those gaps with the other lanes' blocks.  Whole tile rows per lane, so the image
// is bit-identical to the one-stream result.  The second time the same frame description comes
// in, the launches are captured into a CUDA graph, which is replayed from then on.
// tiles: instead of tile rows, the tile map of `tiles` (always written in frame layout, one lane).
// hotF32 / hotU8: BandView::hot_* (the output must then be in frame layout, or the whole frame).
int render_bands(McContext* ctx, int first, int stride, float4* outF32, uchar4* outU8, cudaStream_t stream,
                 bool frameLayout = false, const BandSpec* tiles = nullptr, float4* hotF32 = nullptr, uchar4* hotU8 = nullptr) {
    const DevFrame& f = ctx->prep.frame;
    const int nRows = tiles ? (tiles->nTiles > 0 ? 1 : 0) : local_tile_rows(f, first, stride);
    const int L = (ctx->isChild || tiles) ? 1 : std::max(1, std::min(ctx->frameLanes, nRows / 2));
    ctx->splitLastRender = 0;
    ctx->graphLastRender = false;
    if (!ctx->isChild && f.soft_on) seed_memo_of(ctx);
    if (stream != ctx->stream && ctx->evUpload) CU_TRY(cudaStreamWaitEvent(stream, ctx->evUpload, 0));
    if (L > 1) {
        const int rc = ensure_lanes(ctx, L - 1);
        if (rc != MC_OK) return rc;
        for (int k = 1; k < L; ++k) inherit_options(ctx->lanes[k - 1], ctx);
    }
    const bool graphable = ctx->useGraphs && !ctx->isChild && nRows > 0 && !ctx->forceAllActive && f.spp <= kBlockThreads &&
                           f.width <= 65535 && f.height <= 65535;
    McContext::GraphKey key;
    std::memset(&key, 0, sizeof(key));
    if (graphable) {
        key.frame = f;
        key.blob = ctx->boxes.p; key.texels = ctx->texels.p; key.outF32 = outF32; key.outU8 = outU8;
        key.blobBytes = static_cast<unsigned int>(ctx->prep.blob.size());
        key.first = first; key.stride = stride; key.lanes = L * 2 + (frameLayout ? 1 : 0);
        key.hotF32 = hotF32; key.hotU8 = hotU8;
        key.aovCoverage = ctx->aov.coverage; key.aovDepth = ctx->aov.depth; key.aovTriId = ctx->aov.tri_id;
        if (tiles) {
            key.tileMap = tiles->map; key.mapVersion = tiles->mapVersion; key.nTiles = tiles->nTiles; key.nHeavy = tiles->nHeavy;
        }
        for (int i = 0; i < 12; ++i) key.optionBits[i] = option_bits(ctx, i);
        key.allocEpoch = g_allocEpoch.load();
        if (ctx->graphExec && key == ctx->graphKey) {
            // the graph skips the tile seeding when the seeds were already in place at capture time
            bool seedsIntact = ctx->graphSeedGens.size() == static_cast<size_t>(L) && ctx->graphSeedGens[0] == ctx->seedGen;
            for (int k = 1; seedsIntact && k < L; ++k) seedsIntact = ctx->graphSeedGens[k] == ctx->lanes[k - 1]->seedGen;
            if (seedsIntact) {
                CU_TRY(cudaEventRecord(ctx->ev0, stream));
                CU_TRY(cudaGraphLaunch(ctx->graphExec, stream));
                CU_TRY(cudaEventRecord(ctx->ev1, stream));
                ctx->stats = McRenderStats{};
                ctx->stats.n_samples = static_cast<int64_t>(f.width) * f.height * f.spp;
                ctx->stats.n_tiles = ctx->graphLaneTiles[0];
                ctx->stats.n_kernel_launches = ctx->graphLaneLaunches[0];
                ctx->chunksLastRender = ctx->graphLaneChunks[0];
                ctx->statsPending = true;
                for (int k = 1; k < L; ++k) {
                    McContext* lane = ctx->lanes[k - 1];
                    lane->stats = McRenderStats{};
                    lane->stats.n_tiles = ctx->graphLaneTiles[k];
                    lane->stats.n_kernel_launches = ctx->graphLaneLaunches[k];
                    lane->chunksLastRender = ctx->graphLaneChunks[k];
                    lane->statsPending = true;
                    lane->graphLastRender = true;
                }
                ctx->splitLastRender = L - 1;
                ctx->graphLastRender = true;
                return MC_OK;
            }
            drop_graph(ctx);
        }
    }
    const bool capture = graphable && ctx->hasCandidate && key == ctx->graphCandidate;
    ctx->hasCandidate = graphable && !capture;
    if (graphable) ctx->graphCandidate = key;
    if (capture) {
        drop_graph(ctx);
        ctx->capturing = true;
        for (int k = 1; k < L; ++k) ctx->lanes[k - 1]->capturing = true;
        cudaError_t e = cudaStreamBeginCapture(stream, cudaStreamCaptureModeRelaxed);
        int rc = e == cudaSuccess ? launch_frame_lanes(ctx, first, stride, L, outF32, outU8, stream, frameLayout, tiles, hotF32, hotU8) : MC_ERR_CUDA;
        cudaGraph_t g = nullptr;
        if (e == cudaSuccess) {
            const cudaError_t e2 = cudaStreamEndCapture(stream, &g);
            if (e2 != cudaSuccess) rc = MC_ERR_CUDA;
        }
        ctx->capturing = false;
        for (int k = 1; k < L; ++k) ctx->lanes[k - 1]->capturing = false;
        const bool reallocated = key.allocEpoch != g_allocEpoch.load();  // cannot happen for an unchanged frame; be safe
        if (rc == MC_OK && g && !reallocated && cudaGraphInstantiate(&ctx->graphExec, g, 0) == cudaSuccess) {
            ctx->graph = g;
            ctx->graphKey = key;
            ctx->graphSeedGens.assign(L, 0);
            ctx->graphLaneLaunches.assign(L, 0);
            ctx->graphLaneChunks.assign(L, 0);
            ctx->graphLaneTiles.assign(L, 0);
            for (int k = 0; k < L; ++k) {
                const McContext* lane = k == 0 ? ctx : ctx->lanes[k - 1];
                ctx->graphSeedGens[k] = lane->seedGen;
                ctx->graphLaneLaunches[k] = lane->stats.n_kernel_launches;
                ctx->graphLaneChunks[k] = lane->chunksLastRender;
                ctx->graphLaneTiles[k] = static_cast<int>(lane->stats.n_tiles);
            }
            return render_bands(ctx, first, stride, outF32, outU8, stream, frameLayout, tiles, hotF32, hotU8);  // replays the graph just made
        }
        // capture failed (an operation that cannot be captured): clear the error state, render directly
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        ctx->graphExec = nullptr;
        ctx->useGraphs = 0;
    }
    CU_TRY(cudaEventRecord(ctx->ev0, stream));
    const int rc = launch_frame_lanes(ctx, first, stride, L, outF32, outU8, stream, frameLayout, tiles, hotF32, hotU8);
    if (rc != MC_OK) return rc;
    if (L > 1) {
        CU_TRY(cudaEventRecord(ctx->ev1, stream));
        ctx->splitLastRender = L - 1;
        ctx->stats.n_samples = static_cast<int64_t>(std::max(f.width, 0)) * std::max(f.height, 0) * f.spp;
    }
    return MC_OK;
}

int finish_stats(McContext* ctx, McRenderStats* out) {
    if (ctx->statsPending) {
        float ms = 0.0f;
        if (!(ctx->isChild && ctx->graphLastRender)) {  // a lane replayed inside its parent's graph has no events of its own
            CU_TRY(cudaEventSynchronize(ctx->ev1));
            CU_TRY(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        }
        ctx->stats.ms_device = ms;
        ctx->stats.ms_primary = ctx->stats.ms_shade = 0.0f;
        for (int c = 0; c < ctx->chunksLastRender && !ctx->graphLastRender; ++c) {
            float a = 0.0f, b = 0.0f;
            CU_TRY(cudaEventElapsedTime(&a, ctx->passEvents[3 * c], ctx->passEvents[3 * c + 1]));
            CU_TRY(cudaEventElapsedTime(&b, ctx->passEvents[3 * c + 1], ctx->passEvents[3 * c + 2]));
            ctx->stats.ms_primary += a;
            ctx->stats.ms_shade += b;
        }
        // (left in countHost by the frame's last kernel or by a copy behind it, before ev1 — for a lane inside its
        // parent's graph: before the parent's ev1, which the parent has waited for by now)
        long long active = 0;
        const unsigned int* counts = static_cast<const unsigned int*>(ctx->countHost.p);
        for (int c = 0; c < ctx->chunksLastRender && counts; ++c) active += counts[c];
        ctx->stats.n_active_pixels = static_cast<int32_t>(std::min<long long>(active, 0x7fffffff));
        ctx->statsPending = false;
        // a frame split over lanes: the lanes ran side by side, so counts add and pass times overlap
        for (int k = 0; k < ctx->splitLastRender; ++k) {
            McRenderStats s{};
            const int rc = finish_stats(ctx->lanes[k], &s);
            if (rc != MC_OK) return rc;
            ctx->stats.n_tiles += s.n_tiles;
            ctx->stats.n_active_pixels += s.n_active_pixels;
            ctx->stats.n_kernel_launches += s.n_kernel_launches;
            ctx->stats.ms_primary = std::max(ctx->stats.ms_primary, s.ms_primary);
            ctx->stats.ms_shade = std::max(ctx->stats.ms_shade, s.ms_shade);
        }
    }
    if (out) *out = ctx->stats;
    return MC_OK;
}

// One cached context per device for the host-facing convenience calls.
std::mutex g_ctxMutex;
std::vector<McContext*> g_ctxByDevice;

int shared_context(int device, McContext** out) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(MC_ERR_NO_DEVICE, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0"));
    if (device < 0 || device >= n) return fail(MC_ERR_INVALID, "device index out of range");
    if (g_ctxByDevice.size() < static_cast<size_t>(n)) g_ctxByDevice.resize(n, nullptr);
    if (!g_ctxByDevice[device]) {
        McContext* c = nullptr;
        const int rc = mcskin_cuda_context_create(device, &c);
        if (rc != MC_OK) return rc;
        g_ctxByDevice[device] = c;
    }
    *out = g_ctxByDevice[device];
    CU_TRY(cudaSetDevice(device));
    return MC_OK;
}

bool is_pinned_host(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}

// A page-locked host range as the device sees it (cudaHostAlloc / torch pin_memory / cudaHostRegisterMapped), or null.
void* device_alias_of_host(void* host) {
    if (!host || !is_pinned_host(host)) return nullptr;
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, host, 0) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return d;
}

// Copies rectangles of the device images to the same places of the host images (both full frames of width W).
int copy_rects_to_host(const std::vector<PixelRect>& rects, int W, const void* dF32, float* hF32, const void* dU8, uint8_t* hU8,
                       cudaStream_t s) {
    for (const PixelRect& r : rects) {
        if (r.w <= 0 || r.h <= 0) continue;
        const size_t at = static_cast<size_t>(r.y) * W + r.x;
        if (hF32)
            CU_TRY(cudaMemcpy2DAsync(hF32 + at * 4, static_cast<size_t>(W) * sizeof(float4), static_cast<const float4*>(dF32) + at,
                                     static_cast<size_t>(W) * sizeof(float4), static_cast<size_t>(r.w) * sizeof(float4), r.h,
                                     cudaMemcpyDeviceToHost, s));
        if (hU8)
            CU_TRY(cudaMemcpy2DAsync(hU8 + at * 4, static_cast<size_t>(W) * sizeof(uchar4), static_cast<const uchar4*>(dU8) + at,
                                     static_cast<size_t>(W) * sizeof(uchar4), static_cast<size_t>(r.w) * sizeof(uchar4), r.h,
                                     cudaMemcpyDeviceToHost, s));
    }
    return MC_OK;
}

// The tiles a primary kernel treats as able to hit (its tileCanHit): tile columns [tx0, tx1] x rows [ty0, ty1],
// empty (returns false) when the figure's rectangle misses the frame.
bool hot_tile_range(const DevFrame& f, int* tx0, int* tx1, int* ty0, int* ty1) {
    if (!f.rect_valid || f.rect_x0 > f.rect_x1 || f.rect_y0 > f.rect_y1) return false;
    if (f.rect_x1 < 0 || f.rect_y1 < 0 || f.rect_x0 >= f.width || f.rect_y0 >= f.height) return false;
    *tx0 = std::max(0, f.rect_x0) / f.tile_size;
    *tx1 = std::min(f.width - 1, f.rect_x1) / f.tile_size;
    *ty0 = std::max(0, f.rect_y0) / f.tile_size;
    *ty1 = std::min(f.height - 1, f.rect_y1) / f.tile_size;
    return true;
}

// Maximal rectangles of a set of tiles (frame tile indices): horizontally adjacent tiles of a tile row merge into
// spans, equal spans of consecutive tile rows merge vertically.
std::vector<PixelRect> tile_rects(const DevFrame& f, std::vector<int32_t> tiles) {
    std::vector<PixelRect> out;
    std::sort(tiles.begin(), tiles.end());
    struct Span { int ty, tx0, tx1; };
    std::vector<Span> spans;
    for (size_t i = 0; i < tiles.size();) {
        const int ty = tiles[i] / f.tiles_x, tx0 = tiles[i] % f.tiles_x;
        int tx1 = tx0;
        size_t j = i + 1;
        while (j < tiles.size() && tiles[j] / f.tiles_x == ty && tiles[j] % f.tiles_x == tx1 + 1) { ++tx1; ++j; }
        spans.push_back({ty, tx0, tx1});
        i = j;
    }
    std::vector<char> used(spans.size(), 0);
    for (size_t i = 0; i < spans.size(); ++i) {
        if (used[i]) continue;
        int tyEnd = spans[i].ty;
        for (size_t j = i + 1; j < spans.size(); ++j) {  // spans are sorted by row, then column
            if (spans[j].ty > tyEnd + 1) break;
            if (!used[j] && spans[j].ty == tyEnd + 1 && spans[j].tx0 == spans[i].tx0 && spans[j].tx1 == spans[i].tx1) {
                used[j] = 1;
                tyEnd = spans[j].ty;
            }
        }
        const int x = spans[i].tx0 * f.tile_size, y = spans[i].ty * f.tile_size;
        out.push_back({x, y, std::min(f.width, (spans[i].tx1 + 1) * f.tile_size) - x, std::min(f.height, (tyEnd + 1) * f.tile_size) - y});
    }
    return out;
}


// Device -> caller's host buffer.  Page-locked destinations (cudaHostAlloc / cudaHostRegister,
// torch pin_memory) are written by DMA directly; pageable ones go through the context's pinned
// staging buffer in two halves so the second DMA overlaps the first memcpy.
int copy_out(McContext* ctx, void* hostDst, const void* devSrc, size_t bytes) {
    if (is_pinned_host(hostDst)) {
        CU_TRY(cudaMemcpyAsync(hostDst, devSrc, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        return MC_OK;  // the caller synchronises the stream
    }
    CU_TRY(ctx->pinned.reserve(bytes));
    const size_t half = (bytes / 2) & ~static_cast<size_t>(4095);
    unsigned char* stage = static_cast<unsigned char*>(ctx->pinned.p);
    const unsigned char* src = static_cast<const unsigned char*>(devSrc);
    CU_TRY(cudaMemcpyAsync(stage, src, half, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaEventRecord(ctx->evCopy, ctx->stream));
    CU_TRY(cudaMemcpyAsync(stage + half, src + half, bytes - half, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaEventSynchronize(ctx->evCopy));
    std::memcpy(hostDst, stage, half);
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    std::memcpy(static_cast<unsigned char*>(hostDst) + half, stage + half, bytes - half);
    return MC_OK;
}

// Runs a single-query launcher: uploads inputs, launches, downloads outputs.
struct Staged {
    McContext* ctx;
    std::vector<void*> temps;
    ~Staged() {
        for (void* p : temps) cudaFree(p);
    }
    int up(const void* host, size_t bytes, void** dev) {
        *dev = nullptr;
        if (bytes == 0) return MC_OK;
        CU_TRY(cudaMalloc(dev, bytes));
        temps.push_back(*dev);
        if (host) CU_TRY(cudaMemcpyAsync(*dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
        return MC_OK;
    }
    int down(void* host, const void* dev, size_t bytes) {
        if (bytes == 0) return MC_OK;
        CU_TRY(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(cudaStreamSynchronize(ctx->stream));
        CU_TRY(cudaGetLastError());
        return MC_OK;
    }
};

int query_setup(const McScene* scene, const McConfig* cfg, int device, int useConfig, float aspect, McContext** ctx) {
    const int rc = shared_context(device, ctx);
    if (rc != MC_OK) return rc;
    std::string err;
    const int prc = prepare_frame(scene, cfg, useConfig, aspect, (*ctx)->prep, err);
    if (prc != MC_OK) return fail(prc, err);
    (*ctx)->hasScene = true;
    if (cfg) (*ctx)->cfg = *cfg;
    return upload_scene(*ctx);
}

}  // namespace

// =============================================================== exported functions
namespace {

// Batches, grouped form (SURVEY.md §8e "one launch renders many skins"): the scenes of a chunk that
// share a frame description — image size, sampling, camera, light, box layout; in a batch of skins
// that is nearly all of them — are rendered by ONE set of launches whose gridDim.y is the scene.
// Each scene has its own boxes, texels, output image, work list and queues (BatchSlice); the tile
// engines are seeded once per launch set (they do not depend on the scene).  Returns MC_OK with
// *handled = false when the frame description needs a path that has no batched form.
// skins: instead of flat scenes, raw RGBA8 atlases (SURVEY.md §8f row 3): the host lays out the boxes of every skin
// from the alpha bytes alone (skin_layout) and uploads the 16 KB atlas; k_slice_skins cuts it into the scene's
// float texel pool on the device (SkinParser::parse, skin_parser.cpp:11-110 + image.cpp:14-21) — a third of
// the bytes per skin over PCIe, and no float conversion on the host.
struct SkinBatchSrc {
    const uint8_t* atlases;
    int w, h;
    const float* poses;   // 12 floats per skin, or one set for all (poseStride 0), or null
    int poseStride;
};

int render_batch_grouped(McContext* ctx, const McScene* scenes, const SkinBatchSrc* skins, int nScenes, const McConfig* cfg,
                         float4* outF32, uchar4* outU8, cudaStream_t stream, bool* handled) {
    *handled = false;
    if (!ctx->batchMode || ctx->shadeMode != 0 || ctx->forceAllActive || nScenes < 2) return MC_OK;
    if (cfg->width <= 0 || cfg->height <= 0 || cfg->tile_size <= 0 || cfg->width > 65535 || cfg->height > 65535) return MC_OK;
    const int spp = std::max(1, cfg->samples_per_pixel);
    if (spp > kBlockThreads) return MC_OK;
    const size_t pixels = static_cast<size_t>(cfg->width) * cfg->height;
    std::string err;
    for (int i = 0; i < 2; ++i)
        if (!ctx->evStage[i]) CU_TRY(cudaEventCreateWithFlags(&ctx->evStage[i], cudaEventDisableTiming));

    // sizes per scene (identical for every scene: they depend on the config only)
    PreparedFrame probe;
    const size_t atlasBytes = skins ? static_cast<size_t>(skins->w) * skins->h * 4 : 0;
    // one skin's staging record: atlas | face table | slicing job
    const size_t skinRecord = (atlasBytes + kSkinMaxFaces * sizeof(SkinFaceSource) + sizeof(SkinSliceJob) + 255) & ~size_t(255);
    McBox skinBoxes[kSkinMaxBoxes];
    SkinFaceSource skinFaces[kSkinMaxFaces];
    uint8_t skinOpaque[kSkinMaxBoxes];
    // the flat scene of skin k of the batch (boxes into `boxes`)
    auto layout_skin = [&](int k, McBox* boxes, SkinFaceSource* faces, int* nFaces, uint8_t* opaque, McScene* sc) {
        const float* pose = skins->poses ? skins->poses + static_cast<size_t>(k) * skins->poseStride : nullptr;
        return skin_layout(skins->atlases + static_cast<size_t>(k) * atlasBytes, skins->w, skins->h, pose, boxes, faces, nFaces, opaque, sc);
    };
    int prc;
    if (skins) {
        McScene sc;
        int nFaces = 0;
        if (layout_skin(0, skinBoxes, skinFaces, &nFaces, skinOpaque, &sc) != MC_OK)
            return fail(MC_ERR_INVALID, "render_skin_batch: atlases must be 64x64 or 64x32 RGBA8");
        const ExternalTexels ext{skinOpaque};
        prc = prepare_frame(&sc, cfg, 1, 0.0f, probe, err, &ext);
    } else {
        prc = prepare_frame(&scenes[0], cfg, 1, 0.0f, probe, err);
    }
    if (prc != MC_OK) return fail(prc, err);
    const DevFrame& f0 = probe.frame;
    const size_t slotCap = static_cast<size_t>(f0.tiles_x) * f0.tiles_y * f0.tile_size * f0.tile_size;
    const size_t paths = slotCap * f0.spp;
    if (paths > 0x7fffff00u) return MC_OK;
    const size_t recordBytes = std::max<size_t>(16, slotCap * f0.spp * f0.draws_per_sample * sizeof(float));
    const size_t entries = paths * static_cast<size_t>(wavefront_max_hits_per_path(f0));  // cannot overflow
    if (entries > 0xffffff00u) return MC_OK;
    const bool aov = aov_on(ctx);
    const size_t waveBytes = (paths * wavefront_bytes_per_path(f0, aov) + entries * wavefront_bytes_per_entry() +
                              wavefront_fixed_bytes(f0) + 16 * 256 + 255) & ~size_t(255);
    const size_t perScene = waveBytes + recordBytes + slotCap * sizeof(uint2);
    int G = std::min<int>(ctx->batchGroup, nScenes);
    G = static_cast<int>(std::max<size_t>(1, std::min<size_t>(G, static_cast<size_t>(ctx->waveBudgetBytes) / std::max<size_t>(1, perScene))));
    if (G < 2) return MC_OK;
    // launch_primary_batch needs the pixel-per-lane kernels; probe with an empty launch description
    {
        const long long tileDraws = static_cast<long long>(f0.tile_size) * f0.tile_size * f0.spp * std::max(1, f0.draws_per_sample);
        if (!(tileDraws < (1ll << 30) && kBlockThreads * f0.spp * f0.draws_per_sample + 624 <= 16384)) return MC_OK;
    }
    constexpr size_t kMaxBlob = kMaxSceneSmemBytes;
    // blob + texel pool of the largest scene of the batch (a skin scene is ~55 KB)
    size_t sceneStride = 0;
    if (skins)
        sceneStride = ((SceneBlobLayout(kSkinMaxBoxes).bytes() + 255) & ~size_t(255)) +
                      (((static_cast<size_t>(kSkinMaxTexels) + 2) * sizeof(float4h) + 255) & ~size_t(255));
    for (int i = 0; i < nScenes && !skins; ++i) {
        if (scenes[i].n_boxes < 0 || scenes[i].n_texels < 0) return fail(MC_ERR_INVALID, "render_batch: scene has negative counts");
        const size_t blob = (SceneBlobLayout(scenes[i].n_boxes).bytes() + 255) & ~size_t(255);
        if (blob > kMaxBlob) return MC_OK;  // the frame-by-frame path reports the limit
        const size_t tex = ((static_cast<size_t>(scenes[i].n_texels) + 2) * sizeof(float4h) + 255) & ~size_t(255);
        sceneStride = std::max(sceneStride, blob + tex);
    }
    if (sceneStride > (8u << 20)) return MC_OK;
    // per scene: its data, its slice, its AOV view
    const size_t perSceneStage = sceneStride + sizeof(BatchSlice) + sizeof(AovView);
    CU_TRY(ctx->batchScenes.reserve(static_cast<size_t>(G) * perSceneStage));
    CU_TRY(ctx->batchSlots.reserve(static_cast<size_t>(G) * slotCap * sizeof(uint2)));
    CU_TRY(ctx->batchRecords.reserve(static_cast<size_t>(G) * recordBytes));
    CU_TRY(ctx->batchWave.reserve(static_cast<size_t>(G) * waveBytes));
    uint2* const batchSeedMemo = f0.soft_on ? seed_memo_of(ctx) : nullptr;
    CU_TRY(ctx->batchCounts.reserve(static_cast<size_t>(G) * sizeof(unsigned int)));
    CU_TRY(ctx->tileStates.reserve(std::max<size_t>(16, static_cast<size_t>(f0.tiles_x) * f0.tiles_y * 624 * sizeof(uint32_t) *
                                                            static_cast<size_t>(primary_states_per_tile(f0, f0.tiles_x * f0.tiles_y, 1, ctx->smCount * ctx->primaryBlocksPerSm, 0)))));
    for (int i = 0; i < 2; ++i) CU_TRY(ctx->batchStage[i].reserve(static_cast<size_t>(G) * perSceneStage));
    if (skins) {
        CU_TRY(ctx->batchSkinSrc.reserve(static_cast<size_t>(G) * skinRecord));
        for (int i = 0; i < 2; ++i) CU_TRY(ctx->batchSkinStage[i].reserve(static_cast<size_t>(G) * skinRecord));
        ctx->batchSkinBoxes.resize(static_cast<size_t>(G) * kSkinMaxBoxes);
    }
    if (ctx->batchPreps.size() < static_cast<size_t>(G)) ctx->batchPreps.resize(G);
    ctx->tileSeedValid = false;  // this path seeds the engines itself
    ++ctx->seedGen;

    unsigned char* devScenes = static_cast<unsigned char*>(ctx->batchScenes.p);
    const size_t sliceOffset = static_cast<size_t>(G) * sceneStride;  // slices follow the scene data, AOV views the slices
    const size_t aovOffset = sliceOffset + static_cast<size_t>(G) * sizeof(BatchSlice);
    int stageSlot = 0;
    bool seeded = false;
    int seededStatesPerTile = 0;
    for (int c0 = 0; c0 < nScenes; c0 += G) {
        const int nC = std::min(G, nScenes - c0);
        // (the staging buffers of this slot are free once the copies that last read them are done)
        CU_TRY(cudaEventSynchronize(ctx->evStage[stageSlot]));
        unsigned char* skinStage = skins ? static_cast<unsigned char*>(ctx->batchSkinStage[stageSlot].p) : nullptr;
        unsigned char* devSkin = static_cast<unsigned char*>(ctx->batchSkinSrc.p);
        for (int i = 0; i < nC; ++i) {
            if (skins) {
                // atlas, face table and slicing job of skin i into its staging record; the boxes stay on the host
                unsigned char* rec = skinStage + static_cast<size_t>(i) * skinRecord;
                SkinFaceSource* faces = reinterpret_cast<SkinFaceSource*>(rec + atlasBytes);
                SkinSliceJob* job = reinterpret_cast<SkinSliceJob*>(rec + atlasBytes + kSkinMaxFaces * sizeof(SkinFaceSource));
                McScene sc;
                int nFaces = 0;
                McBox* boxes = ctx->batchSkinBoxes.data() + static_cast<size_t>(i) * kSkinMaxBoxes;
                if (layout_skin(c0 + i, boxes, faces, &nFaces, skinOpaque, &sc) != MC_OK)
                    return fail(MC_ERR_INVALID, "render_skin_batch: atlases must be 64x64 or 64x32 RGBA8");
                std::memcpy(rec, skins->atlases + static_cast<size_t>(c0 + i) * atlasBytes, atlasBytes);
                const ExternalTexels ext{skinOpaque};
                prc = prepare_frame(&sc, cfg, 1, 0.0f, ctx->batchPreps[i], err, &ext);
                if (prc != MC_OK) return fail(prc, err);
                const size_t blobBytes = (ctx->batchPreps[i].blob.size() + 255) & ~size_t(255);
                unsigned char* devRec = devSkin + static_cast<size_t>(i) * skinRecord;
                job->atlas = reinterpret_cast<const uchar4*>(devRec);
                job->faces = reinterpret_cast<const SkinFaceSource*>(devRec + atlasBytes);
                job->texels = reinterpret_cast<float4*>(static_cast<unsigned char*>(ctx->batchScenes.p) + static_cast<size_t>(i) * sceneStride + blobBytes);
                job->atlasW = skins->w;
                job->atlasH = skins->h;
                job->nFaces = nFaces;
                job->nTexels = sc.n_texels;
                if (blobBytes + (static_cast<size_t>(sc.n_texels) + 2) * sizeof(float4h) > sceneStride)
                    return fail(MC_ERR_LIMIT, "render_skin_batch: skin scene larger than a skin can be");
                continue;
            }
            prc = prepare_frame(&scenes[c0 + i], cfg, 1, 0.0f, ctx->batchPreps[i], err);
            if (prc != MC_OK) return fail(prc, err);
            if (ctx->batchPreps[i].blob.size() > kMaxBlob ||
                ((ctx->batchPreps[i].blob.size() + 255) & ~size_t(255)) + ctx->batchPreps[i].texels.size() * sizeof(float4h) > sceneStride)
                return fail(MC_ERR_LIMIT, "render_batch: scene larger than its McScene counts imply");
        }
        // groups of equal frame descriptions (and blob sizes), in first-seen order
        std::vector<int> groupOf(nC, -1);
        std::vector<std::vector<int>> groups;
        for (int i = 0; i < nC; ++i) {
            for (size_t g = 0; g < groups.size() && groupOf[i] < 0; ++g) {
                const PreparedFrame& ref = ctx->batchPreps[groups[g][0]];
                if (std::memcmp(&ref.frame, &ctx->batchPreps[i].frame, sizeof(DevFrame)) == 0 &&
                    ref.blob.size() == ctx->batchPreps[i].blob.size())
                    groupOf[i] = static_cast<int>(g);
            }
            if (groupOf[i] < 0) {
                groupOf[i] = static_cast<int>(groups.size());
                groups.emplace_back();
            }
            groups[groupOf[i]].push_back(i);
        }
        // stage: scene data at slot i (chunk-local index), slices ordered group by group
        unsigned char* stage = static_cast<unsigned char*>(ctx->batchStage[stageSlot].p);
        BatchSlice* stageSlices = reinterpret_cast<BatchSlice*>(stage + sliceOffset);
        AovView* stageAovs = reinterpret_cast<AovView*>(stage + aovOffset);
        int sliceAt = 0;
        std::vector<int> groupFirstSlice(groups.size(), 0);
        for (size_t g = 0; g < groups.size(); ++g) {
            groupFirstSlice[g] = sliceAt;
            for (int i : groups[g]) {
                const PreparedFrame& pf = ctx->batchPreps[i];
                unsigned char* dst = stage + static_cast<size_t>(i) * sceneStride;
                const size_t blobBytes = (pf.blob.size() + 255) & ~size_t(255);
                std::memcpy(dst, pf.blob.data(), pf.blob.size());
                if (!skins) std::memcpy(dst + blobBytes, pf.texels.data(), pf.texels.size() * sizeof(float4h));
                BatchSlice sl{};
                sl.fp.blob = devScenes + static_cast<size_t>(i) * sceneStride;
                sl.fp.texels = reinterpret_cast<const float4*>(devScenes + static_cast<size_t>(i) * sceneStride + blobBytes);
                sl.fp.blob_bytes = static_cast<unsigned int>(pf.blob.size());
                sl.band.first_tile_row = 0;
                sl.band.tile_row_stride = 1;
                sl.band.n_tile_rows = pf.frame.tiles_y;
                sl.band.out_first_row = 0;
                sl.band.out_row_stride = 1;
                sl.band.out_f32 = outF32 ? outF32 + static_cast<size_t>(c0 + i) * pixels : nullptr;
                sl.band.out_u8 = outU8 ? outU8 + static_cast<size_t>(c0 + i) * pixels : nullptr;
                AovView av{};
                av.planes = aov_at(ctx->aov, static_cast<size_t>(c0 + i) * pixels);
                sl.list.count = static_cast<unsigned int*>(ctx->batchCounts.p) + i;
                sl.list.slot_pixel = static_cast<uint2*>(ctx->batchSlots.p) + static_cast<size_t>(i) * slotCap;
                sl.list.records = reinterpret_cast<float*>(static_cast<unsigned char*>(ctx->batchRecords.p) + static_cast<size_t>(i) * recordBytes);
                sl.list.capacity = static_cast<unsigned int>(slotCap);
                sl.list.count_host = nullptr;
                // few blocks per scene: a launch has gridDim.y scenes to fill the machine with
                const int gridX = std::max(2, (ctx->smCount * ctx->shadeBlocksPerSm + nC - 1) / nC);
                if (!wavefront_carve(pf.frame, static_cast<unsigned char*>(ctx->batchWave.p) + static_cast<size_t>(i) * waveBytes,
                                     waveBytes, static_cast<unsigned int>(paths), static_cast<unsigned int>(entries), gridX, &sl.wave, aov ? &av : nullptr))
                    return MC_OK;  // (cannot happen: the sizes depend on the config only) frame-by-frame path instead
                sl.wave.seedMemo = batchSeedMemo;
                stageAovs[sliceAt] = av;
                stageSlices[sliceAt++] = sl;
            }
        }
        const size_t usedScenes = static_cast<size_t>(nC) * sceneStride;
        if (skins) {
            // only the box records of every scene go up (one strided copy), and the raw atlases; the texel pools are cut on the device
            const size_t blobMax = (SceneBlobLayout(kSkinMaxBoxes).bytes() + 255) & ~size_t(255);
            CU_TRY(cudaMemcpy2DAsync(devScenes, sceneStride, stage, sceneStride, blobMax, nC, cudaMemcpyHostToDevice, stream));
            CU_TRY(cudaMemcpyAsync(devSkin, skinStage, static_cast<size_t>(nC) * skinRecord, cudaMemcpyHostToDevice, stream));
            launch_slice_skins(devSkin, skinRecord, atlasBytes + kSkinMaxFaces * sizeof(SkinFaceSource), nC, stream);
        } else {
            CU_TRY(cudaMemcpyAsync(devScenes, stage, usedScenes, cudaMemcpyHostToDevice, stream));
        }
        CU_TRY(cudaMemcpyAsync(devScenes + sliceOffset, stage + sliceOffset, static_cast<size_t>(nC) * sizeof(BatchSlice),
                               cudaMemcpyHostToDevice, stream));
        if (aov)
            CU_TRY(cudaMemcpyAsync(devScenes + aovOffset, stage + aovOffset, static_cast<size_t>(nC) * sizeof(AovView),
                                   cudaMemcpyHostToDevice, stream));
        CU_TRY(cudaEventRecord(ctx->evStage[stageSlot], stream));
        stageSlot ^= 1;
        const BatchSlice* devSlices = reinterpret_cast<const BatchSlice*>(devScenes + sliceOffset);
        const AovView* devAovs = aov ? reinterpret_cast<const AovView*>(devScenes + aovOffset) : nullptr;
        for (size_t g = 0; g < groups.size(); ++g) {
            const int nS = static_cast<int>(groups[g].size());
            const BatchSlice* gs = devSlices + groupFirstSlice[g];
            const AovView* gAov = devAovs ? devAovs + groupFirstSlice[g] : nullptr;
            const BatchSlice& first = stageSlices[groupFirstSlice[g]];
            const DevFrame& f = ctx->batchPreps[groups[g][0]].frame;
            launch_batch_reset(gs, nS, stream);
            if (gAov) launch_aov_defaults(f, first.band, McAovTargets{}, gAov, nS, stream);
            const int build = f.rng_mode ? 2 : (f.any_rotated ? 0 : 1);  // (equal frame descriptions: equal for the whole group)
            // the engines are seeded once per batch — same image geometry for every scene — unless a group is small enough
            // for its tiles to be split over blocks, which changes what is kept per tile
            const int primaryTarget = ctx->smCount * ctx->primaryBlocksPerSm;
            const int statesPerTile = primary_states_per_tile(f, f.tiles_x * f.tiles_y, nS, primaryTarget, 0);
            const bool seedNow = !seeded || statesPerTile != seededStatesPerTile;
            uint32_t* const states = static_cast<uint32_t*>(ctx->tileStates.p);
            const bool launched =
                build == 2 ? counter::launch_primary_batch(f, first.band, states, seedNow, gs, nS, first.fp.blob_bytes, primaryTarget, stream)
                : build == 1 ? plain::launch_primary_batch(f, first.band, states, seedNow, gs, nS, first.fp.blob_bytes, primaryTarget, stream)
                             : launch_primary_batch(f, first.band, states, seedNow, gs, nS, first.fp.blob_bytes, primaryTarget, stream);
            if (!launched) return MC_OK;  // no batched primary kernel for this frame description: frame-by-frame path instead
            seeded = true;
            seededStatesPerTile = statesPerTile;
            int launches = 0;
            if (build == 2) counter::launch_wavefront(f, first.fp, first.band, first.list, first.wave, nullptr, stream, &launches, gs, nS, nullptr, gAov);
            else if (build == 1) plain::launch_wavefront(f, first.fp, first.band, first.list, first.wave, nullptr, stream, &launches, gs, nS, nullptr, gAov);
            else launch_wavefront(f, first.fp, first.band, first.list, first.wave, nullptr, stream, &launches, gs, nS, nullptr, gAov);
        }
        CU_TRY(cudaGetLastError());
    }
    *handled = true;
    return MC_OK;
}

}  // namespace

extern "C" {

int32_t mcskin_cuda_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int32_t mcskin_cuda_context_create(int32_t device, McContext** out) {
    if (!out) return fail(MC_ERR_INVALID, "context_create: out is null");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(MC_ERR_NO_DEVICE, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0"));
    }
    if (device < 0 || device >= n) return fail(MC_ERR_INVALID, "device index out of range");
    CU_TRY(cudaSetDevice(device));
    std::unique_ptr<McContext> ctx(new McContext());
    ctx->device = device;
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    ctx->smCount = prop.multiProcessorCount;
    CU_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CU_TRY(cudaEventCreate(&ctx->ev0));
    CU_TRY(cudaEventCreate(&ctx->ev1));
    CU_TRY(cudaEventCreateWithFlags(&ctx->evCopy, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&ctx->evPrimaryDone, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&ctx->evFrameDone, cudaEventDisableTiming));
    CU_TRY(cudaStreamCreateWithFlags(&ctx->copyStream, cudaStreamNonBlocking));
    CU_TRY(cudaEventCreateWithFlags(&ctx->evUpload, cudaEventDisableTiming));
    if (const char* v = std::getenv("MCSKIN_FORCE_ALL_ACTIVE")) ctx->forceAllActive = std::atoi(v);
    if (const char* v = std::getenv("MCSKIN_HEAVY_TILES")) ctx->heavyTilesPerSm = std::max(0, std::atoi(v));
    if (const char* v = std::getenv("MCSKIN_PRIMARY_BLOCKS")) ctx->primaryBlocksPerSm = std::max(0, std::atoi(v));
    if (const char* v = std::getenv("MCSKIN_WAVE_QUEUE_PCT")) ctx->waveQueuePct = std::max(0, std::atoi(v));
    if (const char* v = std::getenv("MCSKIN_BATCH_GROUP")) ctx->batchGroup = std::min(4096, std::max(1, std::atoi(v)));
    if (const char* v = std::getenv("MCSKIN_BATCH_MODE")) ctx->batchMode = std::atoi(v) != 0;
    if (const char* v = std::getenv("MCSKIN_GRAPHS")) ctx->useGraphs = std::atoi(v) != 0;
    if (const char* v = std::getenv("MCSKIN_STAGED_COPY")) ctx->stagedCopyOut = std::atoi(v) != 0;
    if (const char* v = std::getenv("MCSKIN_SEED_MEMO")) ctx->shadowSeedMemo = std::atoi(v) != 0;
    if (const char* v = std::getenv("MCSKIN_OVERLAP_COPY")) ctx->overlapCopyOut = std::min(2, std::max(0, std::atoi(v)));
    if (const char* v = std::getenv("MCSKIN_FRAME_LANES")) ctx->frameLanes = std::min(8, std::max(1, std::atoi(v)));
    if (const char* v = std::getenv("MCSKIN_CACHE_TILE_SEEDS")) ctx->cacheTileSeeds = std::atoi(v) != 0;
    if (const char* v = std::getenv("MCSKIN_SHADE_BLOCKS")) ctx->shadeBlocksPerSm = std::max(1, std::atoi(v));
    if (const char* v = std::getenv("MCSKIN_SOFT_BLOCKS")) ctx->softBlocksPerSm = std::max(1, std::atoi(v));
    if (const char* v = std::getenv("MCSKIN_SHADE_MODE")) ctx->shadeMode = std::min(2, std::max(0, std::atoi(v)));
    *out = ctx.release();
    return MC_OK;
}

void mcskin_cuda_context_destroy(McContext* ctx) {
    if (!ctx) return;
    for (McContext* lane : ctx->lanes) mcskin_cuda_context_destroy(lane);
    ctx->lanes.clear();
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (DevBuf* b : {&ctx->boxes, &ctx->texels, &ctx->count, &ctx->slotPixel, &ctx->records, &ctx->imgF32, &ctx->imgU8,
                      &ctx->scratchIn, &ctx->scratchOut, &ctx->countLog, &ctx->wave, &ctx->tileStates, &ctx->tileMap,
                      &ctx->blockTimes})
        b->release();
    ctx->pinned.release();
    ctx->countHost.release();
    ctx->sceneStage.release();
    ctx->seedMemo.release();
    ctx->stageF32.release();
    ctx->stageU8.release();
    for (cudaEvent_t e : ctx->pieceEvents) cudaEventDestroy(e);
    ctx->pieceEvents.clear();
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->evCopy) cudaEventDestroy(ctx->evCopy);
    if (ctx->evPrimaryDone) cudaEventDestroy(ctx->evPrimaryDone);
    if (ctx->evFrameDone) cudaEventDestroy(ctx->evFrameDone);
    for (int i = 0; i < 2; ++i) {
        if (ctx->evStage[i]) cudaEventDestroy(ctx->evStage[i]);
        ctx->batchStage[i].release();
    }
    for (DevBuf* b : {&ctx->batchScenes, &ctx->batchSlots, &ctx->batchRecords, &ctx->batchWave, &ctx->batchCounts, &ctx->batchSkinSrc,
                      &ctx->aovPlanes}) b->release();
    for (int i = 0; i < 2; ++i) ctx->batchSkinStage[i].release();
    if (ctx->copyStream) cudaStreamDestroy(ctx->copyStream);
    if (ctx->evUpload) cudaEventDestroy(ctx->evUpload);
    if (ctx->graphExec) cudaGraphExecDestroy(ctx->graphExec);
    if (ctx->graph) cudaGraphDestroy(ctx->graph);
    for (cudaEvent_t e : ctx->passEvents) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int32_t mcskin_cuda_context_set_option(McContext* ctx, const char* name, int64_t value) {
    if (!ctx || !name) return fail(MC_ERR_INVALID, "set_option: null argument");
    const std::string k(name);
    if (k == "force_all_active") ctx->forceAllActive = value != 0;
    else if (k == "record_budget_bytes") ctx->recordBudgetBytes = std::max<int64_t>(1, value);
    else if (k == "shade_blocks_per_sm") ctx->shadeBlocksPerSm = static_cast<int>(std::max<int64_t>(1, value));
    else if (k == "soft_blocks_per_sm") ctx->softBlocksPerSm = static_cast<int>(std::max<int64_t>(1, value));
    else if (k == "primary_blocks_per_sm") ctx->primaryBlocksPerSm = static_cast<int>(std::max<int64_t>(0, value));
    else if (k == "heavy_tiles_per_sm") ctx->heavyTilesPerSm = static_cast<int>(std::max<int64_t>(0, value));
    else if (k == "batch_lanes") ctx->batchLanes = static_cast<int>(std::min<int64_t>(16, std::max<int64_t>(1, value)));
    else if (k == "batch_group") ctx->batchGroup = static_cast<int>(std::min<int64_t>(4096, std::max<int64_t>(1, value)));
    else if (k == "batch_mode") ctx->batchMode = value != 0;
    else if (k == "shade_mode") ctx->shadeMode = static_cast<int>(std::min<int64_t>(2, std::max<int64_t>(0, value)));
    else if (k == "debug_primary_timing") ctx->debugPrimaryTiming = value != 0;
    else if (k == "wave_queue_pct") ctx->waveQueuePct = static_cast<int>(std::min<int64_t>(100000, std::max<int64_t>(0, value)));
    else if (k == "frame_lanes") ctx->frameLanes = static_cast<int>(std::min<int64_t>(8, std::max<int64_t>(1, value)));
    else if (k == "cache_tile_seeds") ctx->cacheTileSeeds = value != 0;
    else if (k == "use_graphs") ctx->useGraphs = value != 0;
    else if (k == "overlap_copy_out") ctx->overlapCopyOut = static_cast<int>(std::min<int64_t>(2, std::max<int64_t>(0, value)));
    else if (k == "wave_budget_bytes") ctx->waveBudgetBytes = std::max<int64_t>(1 << 20, value);
    else if (k == "staged_copy_out") ctx->stagedCopyOut = value != 0;
    else if (k == "shadow_seed_memo") ctx->shadowSeedMemo = value != 0;
    else return fail(MC_ERR_INVALID, "set_option: unknown option " + k);
    return MC_OK;
}

int32_t mcskin_cuda_context_set_scene(McContext* ctx, const McScene* scene, const McConfig* cfg) {
    if (!ctx || !scene || !cfg) return fail(MC_ERR_INVALID, "set_scene: null argument");
    CU_TRY(cudaSetDevice(ctx->device));
    std::string err;
    const int rc = prepare_frame(scene, cfg, 1, 0.0f, ctx->prep, err);
    if (rc != MC_OK) return fail(rc, err);
    ctx->cfg = *cfg;
    ctx->hasScene = true;
    return upload_scene(ctx);
}

int32_t mcskin_cuda_band_rows(const McConfig* cfg, int32_t first, int32_t stride) {
    if (!cfg || cfg->width <= 0 || cfg->height <= 0 || cfg->tile_size <= 0) return 0;
    DevFrame f{};
    f.width = cfg->width;
    f.height = cfg->height;
    f.tile_size = cfg->tile_size;
    f.tiles_x = (cfg->width + cfg->tile_size - 1) / cfg->tile_size;
    f.tiles_y = (cfg->height + cfg->tile_size - 1) / cfg->tile_size;
    return band_pixel_rows(f, first, stride);
}

int32_t mcskin_cuda_context_render_bands(McContext* ctx, int32_t first, int32_t stride, void* dOutF32, void* dOutU8,
                                         void* stream) {
    if (!ctx || !ctx->hasScene) return fail(MC_ERR_INVALID, "render_bands: no scene set");
    if (stride <= 0 || first < 0) return fail(MC_ERR_INVALID, "render_bands: bad partition");
    CU_TRY(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return render_bands(ctx, first, stride, static_cast<float4*>(dOutF32), static_cast<uchar4*>(dOutU8), s);
}

int32_t mcskin_cuda_context_render_rows_into_frame(McContext* ctx, int32_t first, int32_t stride, void* dFrameF32,
                                                    void* dFrameU8, void* stream) {
    if (!ctx || !ctx->hasScene) return fail(MC_ERR_INVALID, "render_rows_into_frame: no scene set");
    if (stride <= 0 || first < 0) return fail(MC_ERR_INVALID, "render_rows_into_frame: bad partition");
    CU_TRY(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    return render_bands(ctx, first, stride, static_cast<float4*>(dFrameF32), static_cast<uchar4*>(dFrameU8), s, true);
}

// Validates a tile list, orders it (tiles the figure's rectangle touches first), uploads it when it changed and
// describes it for render_bands.  *empty: nothing to render.
static int prepare_tile_map(McContext* ctx, const int32_t* tiles, int32_t nTiles, cudaStream_t s, BandSpec* spec, bool* empty) {
    const DevFrame& f = ctx->prep.frame;
    const bool sameList = ctx->tileMapVersion != 0 && ctx->tileMapHost.size() == static_cast<size_t>(nTiles) &&
                          (nTiles == 0 || std::memcmp(ctx->tileMapHost.data(), tiles, sizeof(int32_t) * nTiles) == 0);
    // the heavy-first order depends on the figure's screen rectangle and the tile grid
    const bool sameOrder = sameList && f.rect_valid == ctx->tileMapFrame.rect_valid && f.rect_x0 == ctx->tileMapFrame.rect_x0 &&
                           f.rect_y0 == ctx->tileMapFrame.rect_y0 && f.rect_x1 == ctx->tileMapFrame.rect_x1 &&
                           f.rect_y1 == ctx->tileMapFrame.rect_y1 && f.tiles_x == ctx->tileMapFrame.tiles_x &&
                           f.tiles_y == ctx->tileMapFrame.tiles_y && f.tile_size == ctx->tileMapFrame.tile_size &&
                           f.width == ctx->tileMapFrame.width && f.height == ctx->tileMapFrame.height;
    if (!sameOrder) {
        const long long total = static_cast<long long>(f.tiles_x) * f.tiles_y;
        std::vector<unsigned char> seen(static_cast<size_t>(std::max<long long>(total, 0)), 0);
        std::vector<int32_t> heavy, light;
        for (int i = 0; i < nTiles; ++i) {
            const int id = tiles[i];
            if (id < 0 || id >= total) return fail(MC_ERR_INVALID, "render_tiles: tile index out of range");
            if (seen[id]) return fail(MC_ERR_INVALID, "render_tiles: tile listed twice");
            seen[id] = 1;
            const int ty = id / f.tiles_x, tx = id - ty * f.tiles_x;
            const int x = tx * f.tile_size, y = ty * f.tile_size;
            const int w = std::min(f.tile_size, f.width - x), h = std::min(f.tile_size, f.height - y);
            // the primary kernels' own test (tileCanHit)
            const bool canHit = !f.rect_valid || !(x > f.rect_x1 || x + w - 1 < f.rect_x0 || y > f.rect_y1 || y + h - 1 < f.rect_y0);
            (canHit ? heavy : light).push_back(id);
        }
        ctx->tileMapHost.assign(tiles, tiles + nTiles);
        ctx->tileMapHeavy = static_cast<int>(heavy.size());
        ctx->tileMapOrdered = heavy;
        ctx->tileMapOrdered.insert(ctx->tileMapOrdered.end(), light.begin(), light.end());
        ctx->tileMapLightRects = tile_rects(f, light);
        ctx->tileMapFrame = f;
        if (nTiles > 0) {
            CU_TRY(ctx->tileMap.reserve(sizeof(int32_t) * static_cast<size_t>(nTiles)));
            // (pageable source: staged before the call returns; ordered after the previous frame's kernels on `s`)
            CU_TRY(cudaMemcpyAsync(ctx->tileMap.p, ctx->tileMapOrdered.data(), sizeof(int32_t) * nTiles, cudaMemcpyHostToDevice, s));
        }
        ++ctx->tileMapVersion;
    }
    *empty = nTiles == 0;
    if (nTiles == 0) {
        ctx->stats = McRenderStats{};
        ctx->statsPending = false;
        return MC_OK;
    }
    spec->map = static_cast<const int*>(ctx->tileMap.p);
    spec->nTiles = nTiles;
    spec->nHeavy = ctx->tileMapHeavy;
    spec->mapVersion = ctx->tileMapVersion;
    return MC_OK;
}

int32_t mcskin_cuda_context_render_tiles_into_frame(McContext* ctx, const int32_t* tiles, int32_t nTiles, void* dFrameF32,
                                                     void* dFrameU8, void* stream) {
    if (!ctx || !ctx->hasScene) return fail(MC_ERR_INVALID, "render_tiles_into_frame: no scene set");
    if (nTiles < 0 || (nTiles > 0 && !tiles)) return fail(MC_ERR_INVALID, "render_tiles_into_frame: bad tile list");
    CU_TRY(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    BandSpec spec;
    bool empty = false;
    const int rc = prepare_tile_map(ctx, tiles, nTiles, s, &spec, &empty);
    if (rc != MC_OK || empty) return rc;
    return render_bands(ctx, 0, 1, static_cast<float4*>(dFrameF32), static_cast<uchar4*>(dFrameU8), s, true, &spec);
}

// The per-frame call of a rank whose scene lives on the CPU and whose result goes to a host image every rank of the
// box shares: upload, this rank's tiles, wait.  The image must be page-locked and mapped (mcskin_cuda_host_register,
// cudaHostAlloc, torch pin_memory).  Tiles the figure's rectangle touches are stored by the kernels straight into it;
// the others go to a device image and leave by DMA, in a few rectangles, once the primary pass is done.
// Asynchronous part of a tile set rendered to a host image: launches on the context's stream (and its copy stream).
// Page-locked, mapped host images take the two-destination route (see render_host); any other host memory gets the
// tiles from a device frame, rectangle by rectangle, after the frame's kernels.
static int launch_tiles_to_host(McContext* ctx, const int32_t* tiles, int32_t nTiles, float* hostF32, uint8_t* hostU8) {
    const DevFrame& f = ctx->prep.frame;
    void* aliasF32 = device_alias_of_host(hostF32);
    void* aliasU8 = device_alias_of_host(hostU8);
    const bool mappedHost = (!hostF32 || aliasF32) && (!hostU8 || aliasU8);
    BandSpec spec;
    bool empty = false;
    int rc = prepare_tile_map(ctx, tiles, nTiles, ctx->stream, &spec, &empty);
    if (rc != MC_OK || empty) return rc;
    const bool classified = !ctx->forceAllActive && f.spp <= kBlockThreads;
    const size_t pixels = static_cast<size_t>(f.width) * f.height;
    if (!mappedHost) {
        if (hostF32) CU_TRY(ctx->imgF32.reserve(pixels * sizeof(float4)));
        if (hostU8) CU_TRY(ctx->imgU8.reserve(pixels * sizeof(uchar4)));
        rc = render_bands(ctx, 0, 1, hostF32 ? static_cast<float4*>(ctx->imgF32.p) : nullptr,
                          hostU8 ? static_cast<uchar4*>(ctx->imgU8.p) : nullptr, ctx->stream, true, &spec);
        if (rc != MC_OK) return rc;
        const std::vector<PixelRect> all = tile_rects(f, ctx->tileMapOrdered);
        return copy_rects_to_host(all, f.width, ctx->imgF32.p, hostF32, ctx->imgU8.p, hostU8, ctx->stream);
    }
    const bool dual = ctx->overlapCopyOut >= 2 && classified && !ctx->tileMapLightRects.empty();
    if (dual) {
        if (hostF32) CU_TRY(ctx->imgF32.reserve(pixels * sizeof(float4)));
        if (hostU8) CU_TRY(ctx->imgU8.reserve(pixels * sizeof(uchar4)));
        rc = render_bands(ctx, 0, 1, hostF32 ? static_cast<float4*>(ctx->imgF32.p) : nullptr,
                          hostU8 ? static_cast<uchar4*>(ctx->imgU8.p) : nullptr, ctx->stream, true, &spec,
                          static_cast<float4*>(aliasF32), static_cast<uchar4*>(aliasU8));
        if (rc != MC_OK) return rc;
        CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->evPrimaryDone, 0));
        return copy_rects_to_host(ctx->tileMapLightRects, f.width, ctx->imgF32.p, hostF32, ctx->imgU8.p, hostU8, ctx->copyStream);
    }
    // every tile straight into the host image
    return render_bands(ctx, 0, 1, static_cast<float4*>(aliasF32), static_cast<uchar4*>(aliasU8), ctx->stream, true, &spec);
}
static int finish_tiles_to_host(McContext* ctx) {
    CU_TRY(cudaSetDevice(ctx->device));
    CU_TRY(cudaStreamSynchronize(ctx->copyStream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    for (McContext* lane : ctx->lanes) CU_TRY(cudaStreamSynchronize(lane->stream));
    CU_TRY(cudaGetLastError());
    return MC_OK;
}

// The per-frame call of a rank whose scene lives on the CPU and whose result goes to a host image every rank of the
// box shares: upload, this rank's tiles, wait.  With a page-locked, mapped image (mcskin_cuda_host_register,
// cudaHostAlloc, torch pin_memory) the tiles the figure's rectangle touches are stored by the kernels straight into
// it; the others go to a device image and leave by DMA, in a few rectangles, once the primary pass is done.
int32_t mcskin_cuda_context_render_scene_tiles(McContext* ctx, const McScene* scene, const McConfig* cfg, const int32_t* tiles,
                                                int32_t nTiles, float* hostF32, uint8_t* hostU8, float* msDevice) {
    if (!ctx) return fail(MC_ERR_INVALID, "render_scene_tiles: null context");
    if (aov_on(ctx)) return fail(MC_ERR_INVALID, "render_scene_tiles: writes no AOV planes; switch the context's AOV targets off first");
    if (nTiles < 0 || (nTiles > 0 && !tiles)) return fail(MC_ERR_INVALID, "render_scene_tiles: bad tile list");
    int rc = mcskin_cuda_context_set_scene(ctx, scene, cfg);
    if (rc != MC_OK) return rc;
    if (msDevice) *msDevice = 0.0f;
    rc = launch_tiles_to_host(ctx, tiles, nTiles, hostF32, hostU8);
    if (rc != MC_OK) return rc;
    rc = finish_tiles_to_host(ctx);
    if (rc != MC_OK) return rc;
    if (msDevice && nTiles > 0) CU_TRY(cudaEventElapsedTime(msDevice, ctx->ev0, ctx->ev1));
    return MC_OK;
}

int32_t mcskin_host_copy_rows(void* dst, const void* src, uint64_t dstPitch, uint64_t srcPitch, uint64_t rowBytes, uint64_t rows,
                              int32_t pieces) {
    if (rows == 0 || rowBytes == 0) return MC_OK;
    if (!dst || !src || pieces <= 0 || dstPitch < rowBytes || srcPitch < rowBytes) return fail(MC_ERR_INVALID, "host_copy_rows: bad argument");
    const uint64_t n = std::min<uint64_t>(rows, static_cast<uint64_t>(pieces));
    std::vector<HostCopyJob> jobs;
    for (uint64_t i = 0; i < n; ++i) {
        const uint64_t r0 = rows * i / n, r1 = rows * (i + 1) / n;
        jobs.push_back({nullptr, static_cast<unsigned char*>(dst) + r0 * dstPitch, static_cast<const unsigned char*>(src) + r0 * srcPitch,
                        static_cast<size_t>(dstPitch), static_cast<size_t>(srcPitch), static_cast<size_t>(rowBytes), static_cast<size_t>(r1 - r0)});
    }
    return run_host_copies(0, jobs) ? MC_OK : fail(MC_ERR_CUDA, "host_copy_rows: copy failed");
}

int32_t mcskin_cuda_host_register(void* hostPtr, uint64_t bytes, void** dPtr) {
    if (!hostPtr || bytes == 0) return fail(MC_ERR_INVALID, "host_register: null or empty range");
    CU_TRY(cudaHostRegister(hostPtr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    if (dPtr) {
        *dPtr = nullptr;
        CU_TRY(cudaHostGetDevicePointer(dPtr, hostPtr, 0));
    }
    return MC_OK;
}
int32_t mcskin_cuda_host_unregister(void* hostPtr) {
    if (!hostPtr) return MC_OK;
    CU_TRY(cudaHostUnregister(hostPtr));
    return MC_OK;
}

int32_t mcskin_cuda_device_alloc(int32_t device, uint64_t bytes, void** out) {
    if (!out) return fail(MC_ERR_INVALID, "device_alloc: out is null");
    *out = nullptr;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaMalloc(out, std::max<uint64_t>(bytes, 16)));
    return MC_OK;
}
int32_t mcskin_cuda_device_free(int32_t device, void* ptr) {
    if (!ptr) return MC_OK;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaFree(ptr));
    return MC_OK;
}
int32_t mcskin_cuda_ipc_export(int32_t device, void* ptr, uint8_t handleOut[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    if (!ptr || !handleOut) return fail(MC_ERR_INVALID, "ipc_export: null argument");
    CU_TRY(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    CU_TRY(cudaIpcGetMemHandle(&h, ptr));
    std::memcpy(handleOut, &h, sizeof(h));
    return MC_OK;
}
int32_t mcskin_cuda_ipc_open(int32_t device, const uint8_t handle[64], void** out) {
    if (!handle || !out) return fail(MC_ERR_INVALID, "ipc_open: null argument");
    *out = nullptr;
    CU_TRY(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    CU_TRY(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return MC_OK;
}
int32_t mcskin_cuda_ipc_close(int32_t device, void* ptr) {
    if (!ptr) return MC_OK;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaIpcCloseMemHandle(ptr));
    return MC_OK;
}

int32_t mcskin_cuda_enable_peer_access(int32_t device, int32_t peer) {
    if (device == peer) return MC_OK;
    CU_TRY(cudaSetDevice(device));
    int can = 0;
    CU_TRY(cudaDeviceCanAccessPeer(&can, device, peer));
    if (!can) return fail(MC_ERR_INVALID, "enable_peer_access: device " + std::to_string(device) + " cannot access device " + std::to_string(peer));
    const cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        return MC_OK;
    }
    CU_TRY(e);
    return MC_OK;
}

int32_t mcskin_cuda_peer_signal(int32_t device, void* dFlag, uint32_t value, void* stream) {
    if (!dFlag) return fail(MC_ERR_INVALID, "peer_signal: null flag");
    CU_TRY(cudaSetDevice(device));
    launch_peer_signal(static_cast<unsigned int*>(dFlag), value, static_cast<cudaStream_t>(stream));
    CU_TRY(cudaGetLastError());
    return MC_OK;
}
int32_t mcskin_cuda_peer_wait(int32_t device, const void* dFlags, int32_t n, uint32_t value, void* dTimeout, void* stream) {
    if (n < 0 || n > 1024 || (n > 0 && !dFlags)) return fail(MC_ERR_INVALID, "peer_wait: bad argument");
    CU_TRY(cudaSetDevice(device));
    launch_peer_wait(static_cast<const unsigned int*>(dFlags), n, value, static_cast<unsigned int*>(dTimeout),
                     static_cast<cudaStream_t>(stream));
    CU_TRY(cudaGetLastError());
    return MC_OK;
}

// diagnosis: (entry ns, exit ns, frame tile, part | parts << 16) of every block of the last primary launch of a
// context rendered with "debug_primary_timing" (one lane, no graph); returns the number of records
int32_t mcskin_cuda_context_debug_block_times(McContext* ctx, uint64_t* out, int32_t capacity) {
    if (!ctx || capacity < 0) return fail(MC_ERR_INVALID, "debug_block_times: bad argument");
    CU_TRY(cudaSetDevice(ctx->device));
    CU_TRY(cudaDeviceSynchronize());
    const int n = std::min(ctx->blockTimesCount, capacity);
    if (out && n > 0) CU_TRY(cudaMemcpy(out, ctx->blockTimes.p, static_cast<size_t>(n) * 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return ctx->blockTimesCount;
}

int32_t mcskin_cuda_context_sync(McContext* ctx, McRenderStats* stats) {
    if (!ctx) return fail(MC_ERR_INVALID, "sync: null context");
    CU_TRY(cudaSetDevice(ctx->device));
    const int rc = finish_stats(ctx, stats);
    if (rc != MC_OK) return rc;
    for (McContext* lane : ctx->lanes) {
        CU_TRY(cudaStreamSynchronize(lane->stream));
        lane->statsPending = false;
    }
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    CU_TRY(cudaGetLastError());
    return MC_OK;
}

// A whole frame into PAGEABLE host images (an Image's std::vector<Color>, a numpy array): the dual-destination route
// of render_host with the library's own page-locked staging images in the caller's place, and host threads that move
// every piece on to the caller's memory as soon as it has arrived — the 93 % of a frame that are final after the primary
// pass cross PCIe and the host's memory while the GPU shades; only the figure's tiles are left when the last kernel ends.
// (One copy of the whole image from device memory followed by one memcpy, the route without this, takes ~4 ms at 1080p.)
static int render_host_staged(McContext* ctx, float* outF32, uint8_t* outU8, int tx0, int tx1, int ty0, int ty1, McRenderStats* stats) {
    const DevFrame& f = ctx->prep.frame;
    const size_t pixels = static_cast<size_t>(f.width) * f.height;
    // (page-locked memory is a scarce resource of the host: frames beyond 1 GiB of staging take the plain route)
    if (pixels * ((outF32 ? sizeof(float4) : 0) + (outU8 ? sizeof(uchar4) : 0)) > (size_t(1) << 30)) return MC_ERR_LIMIT;
    if ((outF32 && ctx->stageF32.reserve(pixels * sizeof(float4)) != cudaSuccess) ||
        (outU8 && ctx->stageU8.reserve(pixels * sizeof(uchar4)) != cudaSuccess)) {
        cudaGetLastError();  // (no page-locked memory to be had: the plain route needs none of this size... or fails on its own)
        return MC_ERR_LIMIT;
    }
    void* aliasF32 = outF32 ? device_alias_of_host(ctx->stageF32.p) : nullptr;
    void* aliasU8 = outU8 ? device_alias_of_host(ctx->stageU8.p) : nullptr;
    if ((outF32 && !aliasF32) || (outU8 && !aliasU8)) return MC_ERR_LIMIT;  // (not mapped: the caller takes the plain route)
    int rc = render_bands(ctx, 0, 1, outF32 ? static_cast<float4*>(ctx->imgF32.p) : nullptr,
                          outU8 ? static_cast<uchar4*>(ctx->imgU8.p) : nullptr, ctx->stream, false, nullptr,
                          static_cast<float4*>(aliasF32), static_cast<uchar4*>(aliasU8));
    if (rc != MC_OK) return rc;
    CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->evPrimaryDone, 0));
    for (int k = 0; k < ctx->splitLastRender; ++k)
        CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->lanes[k]->evPrimaryDone, 0));
    const int ts = f.tile_size, W = f.width;
    const int X0 = tx0 * ts, X1 = std::min(f.width, (tx1 + 1) * ts), Y0 = ty0 * ts, Y1 = std::min(f.height, (ty1 + 1) * ts);
    // pieces of about 2 MB of float pixels: whole rows of the four rectangles around the figure's tiles, then of those tiles
    std::vector<PixelRect> light, hot;
    auto cut = [&](std::vector<PixelRect>& into, int x, int y, int w, int h) {
        if (w <= 0 || h <= 0) return;
        const int rowsPerPiece = std::max(1, (2 << 20) / (w * 16));
        for (int r = 0; r < h; r += rowsPerPiece) into.push_back({x, y + r, w, std::min(rowsPerPiece, h - r)});
    };
    cut(light, 0, 0, W, Y0);
    cut(light, 0, Y0, X0, Y1 - Y0);
    cut(light, X1, Y0, W - X1, Y1 - Y0);
    cut(light, 0, Y1, W, f.height - Y1);
    cut(hot, X0, Y0, X1 - X0, Y1 - Y0);
    while (ctx->pieceEvents.size() < light.size()) {
        cudaEvent_t e;
        CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->pieceEvents.push_back(e);
    }
    std::vector<HostCopyJob> jobs;
    auto add_jobs = [&](const PixelRect& r, cudaEvent_t after) {
        const size_t at = static_cast<size_t>(r.y) * W + r.x;
        if (outF32)
            jobs.push_back({after, reinterpret_cast<unsigned char*>(outF32) + at * 16, static_cast<const unsigned char*>(ctx->stageF32.p) + at * 16,
                            static_cast<size_t>(W) * 16, static_cast<size_t>(W) * 16, static_cast<size_t>(r.w) * 16, static_cast<size_t>(r.h)});
        if (outU8)
            jobs.push_back({after, outU8 + at * 4, static_cast<const unsigned char*>(ctx->stageU8.p) + at * 4,
                            static_cast<size_t>(W) * 4, static_cast<size_t>(W) * 4, static_cast<size_t>(r.w) * 4, static_cast<size_t>(r.h)});
    };
    for (size_t i = 0; i < light.size(); ++i) {
        rc = copy_rects_to_host({light[i]}, W, ctx->imgF32.p, outF32 ? static_cast<float*>(ctx->stageF32.p) : nullptr, ctx->imgU8.p,
                                outU8 ? static_cast<uint8_t*>(ctx->stageU8.p) : nullptr, ctx->copyStream);
        if (rc != MC_OK) return rc;
        CU_TRY(cudaEventRecord(ctx->pieceEvents[i], ctx->copyStream));
        add_jobs(light[i], ctx->pieceEvents[i]);
    }
    if (!run_host_copies(ctx->device, jobs)) CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(ctx->copyStream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < ctx->splitLastRender; ++k) CU_TRY(cudaStreamSynchronize(ctx->lanes[k]->stream));
    CU_TRY(cudaGetLastError());
    jobs.clear();
    for (const PixelRect& r : hot) add_jobs(r, nullptr);
    run_host_copies(ctx->device, jobs);
    return finish_stats(ctx, stats);
}

static int render_host(McContext* ctx, const McScene* scene, const McConfig* cfg, int first, int stride,
                       float* outF32, uint8_t* outU8, size_t hostRowOffsetPixels, McRenderStats* stats) {
    (void)hostRowOffsetPixels;
    int rc = mcskin_cuda_context_set_scene(ctx, scene, cfg);
    if (rc != MC_OK) return rc;
    const DevFrame& f = ctx->prep.frame;
    const int rows = band_pixel_rows(f, first, stride);
    const size_t pixels = static_cast<size_t>(rows) * std::max(f.width, 0);
    if (pixels == 0) {
        if (stats) *stats = McRenderStats{};
        return MC_OK;
    }
    if (outF32) CU_TRY(ctx->imgF32.reserve(pixels * sizeof(float4)));
    if (outU8) CU_TRY(ctx->imgU8.reserve(pixels * sizeof(uchar4)));
    // Two destinations (whole frames into page-locked images the device can address): the tiles the figure's screen
    // rectangle touches — the only ones with pixels that are final as late as the frame's last kernel — are written by
    // the kernels straight into the caller's image (a few MB over PCIe, spread over the frame); all other tiles are
    // final after the primary passes and leave the device image by DMA then, next to the shading kernels.  Nothing
    // is left to copy when the last kernel ends.
    int tx0 = 0, tx1 = -1, ty0 = 0, ty1 = -1;
    const bool wholeFrame = first == 0 && stride == 1;
    const bool classified = !ctx->forceAllActive && f.spp <= kBlockThreads;
    void* aliasF32 = (ctx->overlapCopyOut && wholeFrame && classified && outF32) ? device_alias_of_host(outF32) : nullptr;
    void* aliasU8 = (ctx->overlapCopyOut && wholeFrame && classified && outU8) ? device_alias_of_host(outU8) : nullptr;
    const bool dual = ctx->overlapCopyOut >= 2 && wholeFrame && classified && hot_tile_range(f, &tx0, &tx1, &ty0, &ty1) &&
                      (!outF32 || aliasF32) && (!outU8 || aliasU8);
    if (!dual && ctx->stagedCopyOut && ctx->overlapCopyOut >= 2 && wholeFrame && classified && (outF32 || outU8) &&
        !(outF32 && is_pinned_host(outF32)) && !(outU8 && is_pinned_host(outU8)) && hot_tile_range(f, &tx0, &tx1, &ty0, &ty1)) {
        rc = render_host_staged(ctx, outF32, outU8, tx0, tx1, ty0, ty1, stats);
        if (rc != MC_ERR_LIMIT) return rc;
    }
    if (dual) {
        rc = render_bands(ctx, 0, 1, outF32 ? static_cast<float4*>(ctx->imgF32.p) : nullptr,
                          outU8 ? static_cast<uchar4*>(ctx->imgU8.p) : nullptr, ctx->stream, false, nullptr,
                          static_cast<float4*>(aliasF32), static_cast<uchar4*>(aliasU8));
        if (rc != MC_OK) return rc;
        CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->evPrimaryDone, 0));
        for (int k = 0; k < ctx->splitLastRender; ++k)
            CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->lanes[k]->evPrimaryDone, 0));
        const int ts = f.tile_size;
        const int X0 = tx0 * ts, X1 = std::min(f.width, (tx1 + 1) * ts), Y0 = ty0 * ts, Y1 = std::min(f.height, (ty1 + 1) * ts);
        const std::vector<PixelRect> light = {{0, 0, f.width, Y0}, {0, Y1, f.width, f.height - Y1},
                                              {0, Y0, X0, Y1 - Y0}, {X1, Y0, f.width - X1, Y1 - Y0}};
        rc = copy_rects_to_host(light, f.width, ctx->imgF32.p, outF32, ctx->imgU8.p, outU8, ctx->copyStream);
        if (rc != MC_OK) return rc;
        CU_TRY(cudaStreamSynchronize(ctx->copyStream));
        CU_TRY(cudaStreamSynchronize(ctx->stream));
        for (int k = 0; k < ctx->splitLastRender; ++k) CU_TRY(cudaStreamSynchronize(ctx->lanes[k]->stream));
        CU_TRY(cudaGetLastError());
        return finish_stats(ctx, stats);
    }
    rc = render_bands(ctx, first, stride, outF32 ? static_cast<float4*>(ctx->imgF32.p) : nullptr,
                      outU8 ? static_cast<uchar4*>(ctx->imgU8.p) : nullptr, ctx->stream);
    if (rc != MC_OK) return rc;
    // Copy-out overlapped with shading: once the primary passes are done, every pixel outside the
    // figure's screen rectangle is final (93 % of the headline frame), so the whole image starts its
    // way to the host then, next to the shading kernels; when the frame is complete only the
    // rectangle is sent again.  Needs page-locked destinations (DMA straight into the caller's
    // buffers) and a whole frame in one chunk.
    // (and the classifying primary pass: without it every pixel is written by the shading pass)
    const bool overlap = ctx->overlapCopyOut && first == 0 && stride == 1 && f.rect_valid && ctx->chunksLastRender == 1 &&
                         !ctx->forceAllActive && f.spp <= kBlockThreads && f.rect_x0 <= f.rect_x1 && f.rect_y0 <= f.rect_y1 &&
                         (!outF32 || is_pinned_host(outF32)) && (!outU8 || is_pinned_host(outU8));
    if (overlap) {
        CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->evPrimaryDone, 0));
        for (int k = 0; k < ctx->splitLastRender; ++k)
            CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->lanes[k]->evPrimaryDone, 0));
        if (outF32) CU_TRY(cudaMemcpyAsync(outF32, ctx->imgF32.p, pixels * sizeof(float4), cudaMemcpyDeviceToHost, ctx->copyStream));
        if (outU8) CU_TRY(cudaMemcpyAsync(outU8, ctx->imgU8.p, pixels * sizeof(uchar4), cudaMemcpyDeviceToHost, ctx->copyStream));
        CU_TRY(cudaEventRecord(ctx->evFrameDone, ctx->stream));
        CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->evFrameDone, 0));
        const int x0 = std::max(0, f.rect_x0), x1 = std::min(f.width - 1, f.rect_x1);
        const int y0 = std::max(0, f.rect_y0), y1 = std::min(f.height - 1, f.rect_y1);
        if (x0 <= x1 && y0 <= y1) {
            const size_t at = static_cast<size_t>(y0) * f.width + x0;
            const size_t w = static_cast<size_t>(x1 - x0 + 1), h = static_cast<size_t>(y1 - y0 + 1);
            if (outF32)
                CU_TRY(cudaMemcpy2DAsync(outF32 + at * 4, f.width * sizeof(float4), static_cast<float4*>(ctx->imgF32.p) + at,
                                         f.width * sizeof(float4), w * sizeof(float4), h, cudaMemcpyDeviceToHost, ctx->copyStream));
            if (outU8)
                CU_TRY(cudaMemcpy2DAsync(outU8 + at * 4, f.width * sizeof(uchar4), static_cast<uchar4*>(ctx->imgU8.p) + at,
                                         f.width * sizeof(uchar4), w * sizeof(uchar4), h, cudaMemcpyDeviceToHost, ctx->copyStream));
        }
        CU_TRY(cudaStreamSynchronize(ctx->copyStream));
    } else {
        if (outF32) {
            rc = copy_out(ctx, outF32, ctx->imgF32.p, pixels * sizeof(float4));
            if (rc != MC_OK) return rc;
        }
        if (outU8) {
            rc = copy_out(ctx, outU8, ctx->imgU8.p, pixels * sizeof(uchar4));
            if (rc != MC_OK) return rc;
        }
    }
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    CU_TRY(cudaGetLastError());
    return finish_stats(ctx, stats);
}

int32_t mcskin_cuda_render(const McScene* scene, const McConfig* cfg, int32_t device, float* outF32, uint8_t* outU8,
                           McProgressFn progress, void* user, McRenderStats* stats) {
    if (!scene || !cfg) return fail(MC_ERR_INVALID, "render: null scene or config");
    const int32_t totalTiles = mcskin_generate_tiles(cfg->width, cfg->height, cfg->tile_size, nullptr, 0);
    if (totalTiles == 0) {  // tile_renderer.cpp:144-146: nothing to do, no callbacks
        if (stats) *stats = McRenderStats{};
        return MC_OK;
    }
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = shared_context(device, &ctx);
    if (rc != MC_OK) return rc;
    rc = render_host(ctx, scene, cfg, 0, 1, outF32, outU8, 0, stats);
    if (rc != MC_OK) return rc;
    if (progress)
        for (int32_t i = 1; i <= totalTiles; ++i) progress(i, totalTiles, user);
    return MC_OK;
}

int32_t mcskin_cuda_render_aovs(const McScene* scene, const McConfig* cfg, int32_t device, float* outF32, uint8_t* outU8,
                                const McAovTargets* aov, McRenderStats* stats) {
    if (!scene || !cfg) return fail(MC_ERR_INVALID, "render_aovs: null scene or config");
    const size_t pixels = cfg->width > 0 && cfg->height > 0 ? static_cast<size_t>(cfg->width) * cfg->height : 0;
    const McAovTargets want = aov ? *aov : McAovTargets{};
    const int32_t totalTiles = mcskin_generate_tiles(cfg->width, cfg->height, cfg->tile_size, nullptr, 0);
    if (totalTiles == 0) {  // nothing is rendered: every plane keeps its defaults
        if (want.coverage) std::fill(want.coverage, want.coverage + pixels, 0.0f);
        if (want.depth) std::fill(want.depth, want.depth + pixels, 0.0f);
        if (want.tri_id) std::fill(want.tri_id, want.tri_id + pixels, -1);
        if (stats) *stats = McRenderStats{};
        return MC_OK;
    }
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = shared_context(device, &ctx);
    if (rc != MC_OK) return rc;
    CU_TRY(cudaSetDevice(ctx->device));
    CU_TRY(ctx->aovPlanes.reserve(std::max<size_t>(16, pixels * 3 * sizeof(float))));
    float* const base = static_cast<float*>(ctx->aovPlanes.p);
    McAovTargets dev{};
    dev.coverage = want.coverage ? base : nullptr;
    dev.depth = want.depth ? base + pixels : nullptr;
    dev.tri_id = want.tri_id ? reinterpret_cast<int32_t*>(base + 2 * pixels) : nullptr;
    ctx->aov = dev;
    rc = render_host(ctx, scene, cfg, 0, 1, outF32, outU8, 0, stats);
    ctx->aov = McAovTargets{};
    if (rc != MC_OK) return rc;
    // (render_host has synchronised with the frame)
    if (want.coverage) CU_TRY(cudaMemcpyAsync(want.coverage, dev.coverage, pixels * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (want.depth) CU_TRY(cudaMemcpyAsync(want.depth, dev.depth, pixels * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (want.tri_id) CU_TRY(cudaMemcpyAsync(want.tri_id, dev.tri_id, pixels * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    return MC_OK;
}

int32_t mcskin_cuda_context_set_aov_targets(McContext* ctx, const McAovTargets* dTargets) {
    if (!ctx) return fail(MC_ERR_INVALID, "set_aov_targets: null context");
    ctx->aov = dTargets ? *dTargets : McAovTargets{};
    return MC_OK;
}

int32_t mcskin_cuda_render_tile(const McScene* scene, const McConfig* cfg, int32_t device, const McTile* tile,
                                float* imageF32, uint8_t* imageU8) {
    if (!scene || !cfg || !tile) return fail(MC_ERR_INVALID, "render_tile: null argument");
    if (cfg->width <= 0 || cfg->height <= 0) return fail(MC_ERR_INVALID, "render_tile: empty image");
    if (tile->width <= 0 || tile->height <= 0) return MC_OK;
    if (tile->x < 0 || tile->y < 0 || tile->x + tile->width > cfg->width || tile->y + tile->height > cfg->height)
        return fail(MC_ERR_INVALID, "render_tile: tile outside the image");
    // A tile is rendered as a one-tile frame whose pixel origin is the tile's: same RNG seed
    // (tile.y*width + tile.x), same u,v because the frame size stays the full image's.
    // The kernels address tiles on the tile_size grid, so an off-grid or odd-sized tile is
    // only supported when it coincides with a grid tile.
    const int ts = cfg->tile_size;
    if (ts <= 0 || tile->x % ts != 0 || tile->y % ts != 0 ||
        tile->width != std::min(ts, cfg->width - tile->x) || tile->height != std::min(ts, cfg->height - tile->y))
        return fail(MC_ERR_INVALID, "render_tile: tile is not a tile of generateTiles(width, height, tile_size)");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = shared_context(device, &ctx);
    if (rc != MC_OK) return rc;
    rc = mcskin_cuda_context_set_scene(ctx, scene, cfg);
    if (rc != MC_OK) return rc;
    const DevFrame& f = ctx->prep.frame;
    const int tileRow = tile->y / ts;
    const size_t pixels = static_cast<size_t>(tile->height) * f.width;
    CU_TRY(ctx->imgF32.reserve(pixels * sizeof(float4)));
    CU_TRY(ctx->imgU8.reserve(pixels * sizeof(uchar4)));
    // render the whole tile row (cheap) and copy back only the tile's columns
    rc = render_bands(ctx, tileRow, f.tiles_y, static_cast<float4*>(ctx->imgF32.p), static_cast<uchar4*>(ctx->imgU8.p),
                      ctx->stream);
    if (rc != MC_OK) return rc;
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    if (imageF32)
        CU_TRY(cudaMemcpy2D(imageF32 + (static_cast<size_t>(tile->y) * f.width + tile->x) * 4, f.width * sizeof(float4),
                            static_cast<float4*>(ctx->imgF32.p) + tile->x, f.width * sizeof(float4),
                            tile->width * sizeof(float4), tile->height, cudaMemcpyDeviceToHost));
    if (imageU8)
        CU_TRY(cudaMemcpy2D(imageU8 + (static_cast<size_t>(tile->y) * f.width + tile->x) * 4, f.width * sizeof(uchar4),
                            static_cast<uchar4*>(ctx->imgU8.p) + tile->x, f.width * sizeof(uchar4),
                            tile->width * sizeof(uchar4), tile->height, cudaMemcpyDeviceToHost));
    return finish_stats(ctx, nullptr);
}

int32_t mcskin_cuda_render_multi(const McScene* scene, const McConfig* cfg, int32_t nDevices, float* outF32,
                                 uint8_t* outU8, McRenderStats* stats) {
    if (!scene || !cfg) return fail(MC_ERR_INVALID, "render_multi: null scene or config");
    const int avail = mcskin_cuda_device_count();
    if (avail <= 0) return fail(MC_ERR_NO_DEVICE, "no CUDA device");
    if (nDevices <= 0 || nDevices > avail) return fail(MC_ERR_INVALID, "render_multi: bad device count");
    const int32_t totalTiles = mcskin_generate_tiles(cfg->width, cfg->height, cfg->tile_size, nullptr, 0);
    if (totalTiles == 0) {
        if (stats) *stats = McRenderStats{};
        return MC_OK;
    }
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    std::vector<McContext*> ctxs(nDevices, nullptr);
    // every device gets its cost-balanced tile set (mcskin_partition_tiles) and sends it to the caller's image over
    // its own PCIe link; launch everywhere first (asynchronous), then wait
    std::vector<int32_t> tiles(static_cast<size_t>(totalTiles));
    for (int d = 0; d < nDevices; ++d) {
        int rc = shared_context(d, &ctxs[d]);
        if (rc != MC_OK) return rc;
        McContext* ctx = ctxs[d];
        rc = mcskin_cuda_context_set_scene(ctx, scene, cfg);
        if (rc != MC_OK) return rc;
        const int32_t n = mcskin_partition_tiles(scene, cfg, nDevices, d, -1, tiles.data(), totalTiles);
        if (n < 0) return n;
        rc = launch_tiles_to_host(ctx, tiles.data(), n, outF32, outU8);
        if (rc != MC_OK) return rc;
    }
    McRenderStats total{};
    for (int d = 0; d < nDevices; ++d) {
        int rc = finish_tiles_to_host(ctxs[d]);
        if (rc != MC_OK) return rc;
        McRenderStats s{};
        rc = finish_stats(ctxs[d], &s);
        if (rc != MC_OK) return rc;
        total.n_tiles += s.n_tiles;
        total.n_active_pixels += s.n_active_pixels;
        total.n_kernel_launches += s.n_kernel_launches;
        total.ms_device = std::max(total.ms_device, s.ms_device);
        total.ms_primary = std::max(total.ms_primary, s.ms_primary);
        total.ms_shade = std::max(total.ms_shade, s.ms_shade);
    }
    total.n_samples = static_cast<int64_t>(cfg->width) * cfg->height * std::max(1, cfg->samples_per_pixel);
    if (stats) *stats = total;
    return MC_OK;
}

// Batches (SURVEY.md §8e, config C4): scenes are independent frames.  They are spread round-robin
// over a few "lanes" — child contexts with their own stream, scene buffers, work list and queues —
// so that several small frames are in flight at once and nothing synchronises with the host until
// the caller asks.  Lane k renders scenes k, k+L, k+2L, ... in stream order, which is what makes
// reusing its buffers safe.
int32_t mcskin_cuda_context_render_batch(McContext* ctx, const McScene* scenes, int32_t nScenes, const McConfig* cfg,
                                         void* dOutF32, void* dOutU8, void* stream) {
    if (!ctx || !scenes || !cfg || nScenes < 0) return fail(MC_ERR_INVALID, "render_batch: bad argument");
    if (nScenes == 0) return MC_OK;
    CU_TRY(cudaSetDevice(ctx->device));
    const size_t pixels = static_cast<size_t>(std::max(cfg->width, 0)) * std::max(cfg->height, 0);
    cudaStream_t caller = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    {
        bool handled = false;
        const int rc = render_batch_grouped(ctx, scenes, nullptr, nScenes, cfg, static_cast<float4*>(dOutF32), static_cast<uchar4*>(dOutU8),
                                            caller, &handled);
        if (rc != MC_OK) return rc;
        if (handled) {
            ctx->stats = McRenderStats{};
            ctx->statsPending = false;
            return MC_OK;
        }
    }
    const int nLanes = std::min<int>(ctx->batchLanes, nScenes);
    {
        const int rc = ensure_lanes(ctx, nLanes);
        if (rc != MC_OK) return rc;
    }
    // lanes start after whatever the caller's stream did before (e.g. allocating the outputs)
    CU_TRY(cudaEventRecord(ctx->evCopy, caller));
    for (int k = 0; k < nLanes; ++k) {
        McContext* lane = ctx->lanes[k];
        inherit_options(lane, ctx);
        lane->shadeBlocksPerSm = std::max(1, ctx->shadeBlocksPerSm / 2);  // several frames share the SMs
        CU_TRY(cudaStreamWaitEvent(lane->stream, ctx->evCopy, 0));
    }
    for (int i = 0; i < nScenes; ++i) {
        McContext* lane = ctx->lanes[i % nLanes];
        int rc = mcskin_cuda_context_set_scene(lane, &scenes[i], cfg);
        if (rc != MC_OK) return rc;
        lane->aov = aov_at(ctx->aov, static_cast<size_t>(i) * pixels);
        rc = render_bands(lane, 0, 1, dOutF32 ? static_cast<float4*>(dOutF32) + i * pixels : nullptr,
                          dOutU8 ? static_cast<uchar4*>(dOutU8) + i * pixels : nullptr, lane->stream);
        if (rc != MC_OK) return rc;
    }
    // the caller's stream continues once every lane is done
    for (int k = 0; k < nLanes; ++k) {
        CU_TRY(cudaEventRecord(ctx->lanes[k]->evCopy, ctx->lanes[k]->stream));
        CU_TRY(cudaStreamWaitEvent(caller, ctx->lanes[k]->evCopy, 0));
    }
    ctx->stats = McRenderStats{};
    ctx->statsPending = false;
    return MC_OK;
}

// Batches of skins straight from their atlases (SURVEY.md §8f rows 2-3): n RGBA8 atlases (64x64 or 64x32, one
// after the other) -> n images.  The grouped form lays every skin out on the host from its alpha bytes alone
// and cuts the texel pools on the device; frame descriptions without a batched kernel form build the flat scenes
// on the host (mcskin_build_skin_scene) and take render_batch's frame-by-frame path.
int32_t mcskin_cuda_context_render_skin_batch(McContext* ctx, const uint8_t* atlases, int32_t atlasW, int32_t atlasH,
                                              int32_t nSkins, const float* poses12, int32_t poseStride, const McConfig* cfg,
                                              void* dOutF32, void* dOutU8, void* stream) {
    if (!ctx || !atlases || !cfg || nSkins < 0 || poseStride < 0) return fail(MC_ERR_INVALID, "render_skin_batch: bad argument");
    if (!((atlasW == 64 && atlasH == 64) || (atlasW == 64 && atlasH == 32)))
        return fail(MC_ERR_INVALID, "Invalid skin dimensions: " + std::to_string(atlasW) + "x" + std::to_string(atlasH) +
                                        " (expected 64x64 or 64x32)");
    if (nSkins == 0) return MC_OK;
    CU_TRY(cudaSetDevice(ctx->device));
    cudaStream_t caller = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    const SkinBatchSrc src{atlases, atlasW, atlasH, poses12, poses12 ? poseStride : 0};
    bool handled = false;
    int rc = render_batch_grouped(ctx, nullptr, &src, nSkins, cfg, static_cast<float4*>(dOutF32), static_cast<uchar4*>(dOutU8),
                                  caller, &handled);
    if (rc != MC_OK) return rc;
    if (handled) {
        ctx->stats = McRenderStats{};
        ctx->statsPending = false;
        return MC_OK;
    }
    // host-built scenes, a chunk at a time (each needs 52 KB of texels)
    const size_t atlasBytes = static_cast<size_t>(atlasW) * atlasH * 4;
    const int chunk = 64;
    std::vector<McBox> boxes(static_cast<size_t>(chunk) * kSkinMaxBoxes);
    std::vector<float> texels(static_cast<size_t>(chunk) * (kSkinMaxTexels + 16) * 4);
    std::vector<McScene> scenes(chunk);
    const size_t pixels = static_cast<size_t>(std::max(cfg->width, 0)) * std::max(cfg->height, 0);
    for (int c0 = 0; c0 < nSkins; c0 += chunk) {
        const int n = std::min(chunk, nSkins - c0);
        for (int i = 0; i < n; ++i) {
            const float* pose = poses12 ? poses12 + static_cast<size_t>(c0 + i) * poseStride : nullptr;
            rc = mcskin_build_skin_scene(atlases + static_cast<size_t>(c0 + i) * atlasBytes, atlasW, atlasH, pose,
                                         boxes.data() + static_cast<size_t>(i) * kSkinMaxBoxes,
                                         texels.data() + static_cast<size_t>(i) * (kSkinMaxTexels + 16) * 4, &scenes[i]);
            if (rc != MC_OK) return rc;
        }
        const McAovTargets planes = ctx->aov;  // (the chunk's images start c0 images in)
        ctx->aov = aov_at(planes, static_cast<size_t>(c0) * pixels);
        rc = mcskin_cuda_context_render_batch(ctx, scenes.data(), n, cfg,
                                              dOutF32 ? static_cast<float4*>(dOutF32) + static_cast<size_t>(c0) * pixels : nullptr,
                                              dOutU8 ? static_cast<uchar4*>(dOutU8) + static_cast<size_t>(c0) * pixels : nullptr, caller);
        ctx->aov = planes;
        if (rc != MC_OK) return rc;
        // the host arrays are reused by the next chunk: the uploads above are staged synchronously (pageable sources)
    }
    return MC_OK;
}

// A batch sharded by skin over the devices of this process (SURVEY.md §8e, BASELINE config 4): skin i belongs to
// device i mod nDevices, no exchange of any kind.  One host thread per device prepares, stages and launches
// that device's skins chunk by chunk (mcskin_cuda_context_render_batch) and sends every finished chunk's
// images to the caller's host arrays on a copy stream while the next chunk renders.
int32_t mcskin_cuda_render_batch_multi(const McScene* scenes, int32_t nScenes, const McConfig* cfg, int32_t nDevices,
                                       float* outF32, uint8_t* outU8) {
    if (!scenes || !cfg || nScenes < 0) return fail(MC_ERR_INVALID, "render_batch_multi: bad argument");
    const int avail = mcskin_cuda_device_count();
    if (avail <= 0) return fail(MC_ERR_NO_DEVICE, "no CUDA device");
    if (nDevices <= 0 || nDevices > avail) return fail(MC_ERR_INVALID, "render_batch_multi: bad device count");
    if (nScenes == 0 || (!outF32 && !outU8)) return MC_OK;
    if (cfg->width <= 0 || cfg->height <= 0) return MC_OK;
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    std::vector<McContext*> ctxs(nDevices, nullptr);
    for (int d = 0; d < nDevices; ++d) {
        const int rc = shared_context(d, &ctxs[d]);
        if (rc != MC_OK) return rc;
    }
    const size_t pixels = static_cast<size_t>(cfg->width) * cfg->height;
    std::vector<int> rcs(nDevices, MC_OK);
    std::vector<std::string> errs(nDevices);
    auto work = [&](int d) {
        McContext* ctx = ctxs[d];
        auto run = [&]() -> int {
            CU_TRY(cudaSetDevice(d));
            std::vector<McScene> mine;
            std::vector<int> index;
            for (int i = d; i < nScenes; i += nDevices) {
                mine.push_back(scenes[i]);
                index.push_back(i);
            }
            if (mine.empty()) return MC_OK;
            const int chunk = std::max(1, ctx->batchGroup);
            const size_t slots = std::min<size_t>(mine.size(), 2 * static_cast<size_t>(chunk));  // two chunks in flight
            if (outF32) CU_TRY(ctx->imgF32.reserve(slots * pixels * sizeof(float4)));
            if (outU8) CU_TRY(ctx->imgU8.reserve(slots * pixels * sizeof(uchar4)));
            cudaEvent_t copied[2] = {nullptr, nullptr};
            for (auto& e : copied) CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            int rc = MC_OK;
            int half = 0;
            for (size_t c0 = 0; c0 < mine.size() && rc == MC_OK; c0 += chunk, half ^= 1) {
                const int n = static_cast<int>(std::min<size_t>(chunk, mine.size() - c0));
                float4* dF = outF32 ? static_cast<float4*>(ctx->imgF32.p) + static_cast<size_t>(half) * chunk * pixels : nullptr;
                uchar4* dU = outU8 ? static_cast<uchar4*>(ctx->imgU8.p) + static_cast<size_t>(half) * chunk * pixels : nullptr;
                // this half of the image buffer is free once the copies of the chunk before last have left it
                if (cudaStreamWaitEvent(ctx->stream, copied[half], 0) != cudaSuccess) { rc = MC_ERR_CUDA; break; }
                rc = mcskin_cuda_context_render_batch(ctx, mine.data() + c0, n, cfg, dF, dU, ctx->stream);
                if (rc != MC_OK) break;
                if (cudaEventRecord(ctx->evFrameDone, ctx->stream) != cudaSuccess ||
                    cudaStreamWaitEvent(ctx->copyStream, ctx->evFrameDone, 0) != cudaSuccess) { rc = MC_ERR_CUDA; break; }
                for (int k = 0; k < n && rc == MC_OK; ++k) {
                    const size_t dst = static_cast<size_t>(index[c0 + k]) * pixels;
                    if (outF32 && cudaMemcpyAsync(outF32 + dst * 4, dF + static_cast<size_t>(k) * pixels, pixels * sizeof(float4),
                                                  cudaMemcpyDeviceToHost, ctx->copyStream) != cudaSuccess) rc = MC_ERR_CUDA;
                    if (outU8 && cudaMemcpyAsync(outU8 + dst * 4, dU + static_cast<size_t>(k) * pixels, pixels * sizeof(uchar4),
                                                 cudaMemcpyDeviceToHost, ctx->copyStream) != cudaSuccess) rc = MC_ERR_CUDA;
                }
                if (rc == MC_OK && cudaEventRecord(copied[half], ctx->copyStream) != cudaSuccess) rc = MC_ERR_CUDA;
            }
            if (rc == MC_ERR_CUDA && errs[d].empty()) set_last_error(std::string("render_batch_multi: ") + cudaGetErrorString(cudaGetLastError()));
            cudaStreamSynchronize(ctx->stream);
            cudaStreamSynchronize(ctx->copyStream);
            for (auto& e : copied) cudaEventDestroy(e);
            if (rc != MC_OK) return rc;
            CU_TRY(cudaGetLastError());
            return MC_OK;
        };
        rcs[d] = run();
        if (rcs[d] != MC_OK) errs[d] = mcskin_cuda_last_error();  // the message is thread-local: carry it out
    };
    std::vector<std::thread> threads;
    for (int d = 1; d < nDevices; ++d) threads.emplace_back(work, d);
    work(0);
    for (auto& t : threads) t.join();
    for (int d = 0; d < nDevices; ++d)
        if (rcs[d] != MC_OK) return fail(rcs[d], "device " + std::to_string(d) + ": " + errs[d]);
    return MC_OK;
}

// ------------------------------------------------------------------ single-ray entry points
int32_t mcskin_cuda_intersect(const McScene* scene, int32_t device, int32_t box, const McRay* rays, int32_t n,
                              McHit* out) {
    if (n < 0 || (n > 0 && (!rays || !out))) return fail(MC_ERR_INVALID, "intersect: bad argument");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = query_setup(scene, nullptr, device, 0, 1.0f, &ctx);
    if (rc != MC_OK) return rc;
    if (box >= scene->n_boxes) return fail(MC_ERR_INVALID, "intersect: box index out of range");
    Staged st{ctx, {}};
    void *dR, *dO;
    if ((rc = st.up(rays, sizeof(McRay) * n, &dR)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(McHit) * n, &dO)) != MC_OK) return rc;
    launch_intersect(ctx->prep.frame, frame_pointers(ctx), box, static_cast<McRay*>(dR), n, static_cast<McHit*>(dO),
                     ctx->stream);
    return st.down(out, dO, sizeof(McHit) * n);
}

int32_t mcskin_cuda_trace(const McScene* scene, const McConfig* cfg, int32_t device, int32_t useConfig, int32_t depth,
                          const McRay* rays, int32_t n, float* out) {
    if (!cfg || n < 0 || (n > 0 && (!rays || !out))) return fail(MC_ERR_INVALID, "trace: bad argument");
    // the single-query entry points exist to compare against the reference's functions: mt19937 streams only
    if (cfg->rng_mode != MC_RNG_MT19937) return fail(MC_ERR_INVALID, "trace: rng_mode 1 is a mode of the render entry points only");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = query_setup(scene, cfg, device, useConfig, 0.0f, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void *dR, *dO;
    if ((rc = st.up(rays, sizeof(McRay) * n, &dR)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(float4) * n, &dO)) != MC_OK) return rc;
    launch_trace(ctx->prep.frame, frame_pointers(ctx), depth, static_cast<McRay*>(dR), n, static_cast<float4*>(dO),
                 ctx->stream);
    return st.down(out, dO, sizeof(float4) * n);
}

int32_t mcskin_cuda_shade(const McScene* scene, const McConfig* cfg, int32_t device, const McHit* hits,
                          const float* viewDirs, const float* shadowFactors, int32_t n, float* out) {
    if (!cfg || n < 0 || (n > 0 && (!hits || !viewDirs || !out))) return fail(MC_ERR_INVALID, "shade: bad argument");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = query_setup(scene, cfg, device, 1, 0.0f, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void *dH, *dV, *dS = nullptr, *dO;
    if ((rc = st.up(hits, sizeof(McHit) * n, &dH)) != MC_OK) return rc;
    if ((rc = st.up(viewDirs, sizeof(float) * 3 * n, &dV)) != MC_OK) return rc;
    if (shadowFactors && (rc = st.up(shadowFactors, sizeof(float) * n, &dS)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(float4) * n, &dO)) != MC_OK) return rc;
    launch_shade_hits(ctx->prep.frame, frame_pointers(ctx), static_cast<McHit*>(dH), static_cast<float*>(dV),
                      static_cast<float*>(dS), n, static_cast<float4*>(dO), ctx->stream);
    return st.down(out, dO, sizeof(float4) * n);
}

int32_t mcskin_cuda_in_shadow(const McScene* scene, int32_t device, const float* points, const float* normals,
                              const float* lights, int32_t n, int32_t* out) {
    if (n < 0 || (n > 0 && (!points || !normals || !lights || !out))) return fail(MC_ERR_INVALID, "in_shadow: bad argument");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = query_setup(scene, nullptr, device, 0, 1.0f, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void *dP, *dN, *dL, *dO;
    if ((rc = st.up(points, sizeof(float) * 3 * n, &dP)) != MC_OK) return rc;
    if ((rc = st.up(normals, sizeof(float) * 3 * n, &dN)) != MC_OK) return rc;
    if ((rc = st.up(lights, sizeof(float) * 3 * n, &dL)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(int) * n, &dO)) != MC_OK) return rc;
    launch_in_shadow(ctx->prep.frame, frame_pointers(ctx), static_cast<float*>(dP), static_cast<float*>(dN),
                     static_cast<float*>(dL), n, static_cast<int*>(dO), ctx->stream);
    return st.down(out, dO, sizeof(int) * n);
}

int32_t mcskin_cuda_soft_shadow(const McScene* scene, int32_t device, const float* points, const float* normals,
                                const uint32_t* seeds, int32_t samples, int32_t n, float* out) {
    if (n < 0 || (n > 0 && (!points || !normals || !seeds || !out))) return fail(MC_ERR_INVALID, "soft_shadow: bad argument");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = query_setup(scene, nullptr, device, 0, 1.0f, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void *dP, *dN, *dS, *dO;
    if ((rc = st.up(points, sizeof(float) * 3 * n, &dP)) != MC_OK) return rc;
    if ((rc = st.up(normals, sizeof(float) * 3 * n, &dN)) != MC_OK) return rc;
    if ((rc = st.up(seeds, sizeof(uint32_t) * n, &dS)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(float) * n, &dO)) != MC_OK) return rc;
    launch_soft_shadow(ctx->prep.frame, frame_pointers(ctx), static_cast<float*>(dP), static_cast<float*>(dN),
                       static_cast<uint32_t*>(dS), samples, n, static_cast<float*>(dO), ctx->stream);
    return st.down(out, dO, sizeof(float) * n);
}

int32_t mcskin_cuda_ambient_occlusion(const McScene* scene, int32_t device, const float* points, const float* normals,
                                      const uint32_t* seeds, int32_t samples, float radius, int32_t n, float* out) {
    if (n < 0 || (n > 0 && (!points || !normals || !seeds || !out))) return fail(MC_ERR_INVALID, "ambient_occlusion: bad argument");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = query_setup(scene, nullptr, device, 0, 1.0f, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void *dP, *dN, *dS, *dO;
    if ((rc = st.up(points, sizeof(float) * 3 * n, &dP)) != MC_OK) return rc;
    if ((rc = st.up(normals, sizeof(float) * 3 * n, &dN)) != MC_OK) return rc;
    if ((rc = st.up(seeds, sizeof(uint32_t) * n, &dS)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(float) * n, &dO)) != MC_OK) return rc;
    launch_ambient_occlusion(ctx->prep.frame, frame_pointers(ctx), static_cast<float*>(dP), static_cast<float*>(dN),
                             static_cast<uint32_t*>(dS), samples, radius, n, static_cast<float*>(dO), ctx->stream);
    return st.down(out, dO, sizeof(float) * n);
}

int32_t mcskin_cuda_generate_rays(const McScene* scene, int32_t device, float aspect, const float* uv, int32_t n,
                                  McRay* out) {
    if (n < 0 || (n > 0 && (!uv || !out))) return fail(MC_ERR_INVALID, "generate_rays: bad argument");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = query_setup(scene, nullptr, device, 0, aspect, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void *dU, *dO;
    if ((rc = st.up(uv, sizeof(float) * 2 * n, &dU)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(McRay) * n, &dO)) != MC_OK) return rc;
    launch_generate_rays(ctx->prep.frame, static_cast<float*>(dU), n, static_cast<McRay*>(dO), ctx->stream);
    return st.down(out, dO, sizeof(McRay) * n);
}

int32_t mcskin_cuda_background(const McScene* scene, const McConfig* cfg, int32_t device, int32_t useConfig,
                               const float* uv, int32_t n, float* out) {
    if (!cfg || n < 0 || (n > 0 && (!uv || !out))) return fail(MC_ERR_INVALID, "background: bad argument");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = query_setup(scene, cfg, device, useConfig, 0.0f, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void *dU, *dO;
    if ((rc = st.up(uv, sizeof(float) * 2 * n, &dU)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(float4) * n, &dO)) != MC_OK) return rc;
    launch_background(ctx->prep.frame, static_cast<float*>(dU), n, static_cast<float4*>(dO), ctx->stream);
    return st.down(out, dO, sizeof(float4) * n);
}

int32_t mcskin_primary_launch_order(const McScene* scene, const McConfig* cfg, int32_t first, int32_t stride,
                                    int32_t partsHeavy, int32_t partsLight, int32_t* outTile, int32_t* outPart,
                                    int32_t* outParts, int32_t capacity) {
    if (!scene || !cfg || capacity < 0) return fail(MC_ERR_INVALID, "primary_launch_order: bad argument");
    PreparedFrame pf;
    std::string err;
    const int rc = prepare_frame(scene, cfg, 1, 0.0f, pf, err);
    if (rc != MC_OK) return fail(rc, err);
    return primary_launch_order(pf.frame, first, stride, partsHeavy, partsLight, outTile, outPart, outParts, capacity);
}

int32_t mcskin_cuda_fp32_issue_peak(int32_t device, double* out) {
    if (!out) return fail(MC_ERR_INVALID, "fp32_issue_peak: out is null");
    *out = 0.0;
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = shared_context(device, &ctx);
    if (rc != MC_OK) return rc;
    float* sink = nullptr;
    CU_TRY(cudaMalloc(&sink, sizeof(float)));
    const int blocks = ctx->smCount * 8, iters = 1 << 15;
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {  // the first launches warm the clocks up
        CU_TRY(cudaEventRecord(e0, ctx->stream));
        launch_fp32_peak(blocks, iters, sink, ctx->stream);
        CU_TRY(cudaEventRecord(e1, ctx->stream));
        CU_TRY(cudaEventSynchronize(e1));
        float ms = 0.0f;
        CU_TRY(cudaEventElapsedTime(&ms, e0, e1));
        const double ops = static_cast<double>(blocks) * kBlockThreads * iters * 16.0;
        if (ms > 0.0f) best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    CU_TRY(cudaGetLastError());
    *out = best;
    return MC_OK;
}

int32_t mcskin_cuda_powf(int32_t device, const float* x, const float* y, int32_t n, float* out) {
    if (n < 0 || (n > 0 && (!x || !y || !out))) return fail(MC_ERR_INVALID, "powf: bad argument");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = shared_context(device, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void *dX, *dY, *dO;
    if ((rc = st.up(x, sizeof(float) * n, &dX)) != MC_OK) return rc;
    if ((rc = st.up(y, sizeof(float) * n, &dY)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(float) * n, &dO)) != MC_OK) return rc;
    launch_powf(static_cast<float*>(dX), static_cast<float*>(dY), n, static_cast<float*>(dO), ctx->stream);
    return st.down(out, dO, sizeof(float) * n);
}

int32_t mcskin_cuda_sincos(int32_t device, const float* angles, int32_t n, float* outSin, float* outCos) {
    if (n < 0 || (n > 0 && (!angles || !outSin || !outCos))) return fail(MC_ERR_INVALID, "sincos: bad argument");
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = shared_context(device, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void *dA, *dS, *dC;
    if ((rc = st.up(angles, sizeof(float) * n, &dA)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(float) * n, &dS)) != MC_OK) return rc;
    if ((rc = st.up(nullptr, sizeof(float) * n, &dC)) != MC_OK) return rc;
    launch_sincos(static_cast<float*>(dA), n, static_cast<float*>(dS), static_cast<float*>(dC), ctx->stream);
    if ((rc = st.down(outSin, dS, sizeof(float) * n)) != MC_OK) return rc;
    return st.down(outCos, dC, sizeof(float) * n);
}

int32_t mcskin_cuda_aov(const McScene* scene, const McConfig* cfg, int32_t device, int32_t* outTriId) {
    if (!cfg || !outTriId) return fail(MC_ERR_INVALID, "aov: bad argument");
    if (cfg->width <= 0 || cfg->height <= 0) return MC_OK;
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = query_setup(scene, cfg, device, 1, 0.0f, &ctx);
    if (rc != MC_OK) return rc;
    Staged st{ctx, {}};
    void* dO;
    const size_t bytes = sizeof(int32_t) * static_cast<size_t>(cfg->width) * cfg->height;
    if ((rc = st.up(nullptr, bytes, &dO)) != MC_OK) return rc;
    launch_aov(ctx->prep.frame, frame_pointers(ctx), static_cast<int*>(dO), ctx->stream);
    return st.down(outTriId, dO, bytes);
}

// struct sizes, so bindings can check their mirror of the header
void mcskin_cuda_abi_sizes(int32_t* out8) {
    if (!out8) return;
    out8[0] = sizeof(McFaceTex);
    out8[1] = sizeof(McBox);
    out8[2] = sizeof(McScene);
    out8[3] = sizeof(McConfig);
    out8[4] = sizeof(McTile);
    out8[5] = sizeof(McRenderStats);
    out8[6] = sizeof(McRay);
    out8[7] = sizeof(McHit);
}

}  // extern "C"
