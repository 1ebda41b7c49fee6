// frame.cu — a frame on the device: band sizing, the launches of a lane, frames split over lanes, graph capture and
// replay, tile maps.
#include <cstring>
#include "capi_internal.hpp"

FramePointers frame_pointers(const McContext* ctx) {
    return FramePointers{static_cast<const unsigned char*>(ctx->boxes.p), static_cast<const float4*>(ctx->texels.p),
                         static_cast<unsigned int>(ctx->prep.blob.size())};
}

namespace {

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

}  // namespace

// The table of FreshStream::seed_memo, allocated and zeroed the first time a frame with soft shadows comes in (never
// inside a graph capture: the frame that is captured has been rendered once before).  Null when switched off.
uint2* seed_memo_of(McContext* ctx) {
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

namespace {

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

// Tiles a band covers.
long long band_tiles(const DevFrame& f, const BandSpec& spec) {
    return spec.map ? spec.nTiles : static_cast<long long>(local_tile_rows(f, spec.first, spec.stride)) * f.tiles_x;
}

// How a band is rendered: its chunks, the work-list, engine-state and queue sizes they need, and the grid targets of
// the primary pass.
struct BandPlan {
    bool classify;                 // the primary pass lists only pixels that can hit (else every pixel, positionally)
    size_t nUnits, tilesPerUnit;   // units: whole tile rows, or tiles of the map
    size_t slotsPerUnit, recordBytesPerSlot;
    size_t unitsPerChunk, slotCap;
    int nChunks, heavyTarget, primaryTarget;
    size_t statesPerTile;
    size_t wavePaths, waveEntries, waveBytes;  // wavefront queues (shade_mode 0)
};

// Sizes a band of a frame that fits the limits render_bands_lane checks.  No side effects.
BandPlan plan_band(const DevFrame& f, const BandSpec& spec, const McContext& ctx, int lanesInFlight) {
    BandPlan p{};
    const bool mapped = spec.map != nullptr;
    p.classify = !ctx.forceAllActive && f.spp <= kBlockThreads;
    // A band is rendered in chunks of UNITS — whole tile rows, or tiles of the map — so that the worst-case
    // work list of a chunk fits the budget.  Work-list slots a unit can need: every pixel, or, as the
    // classifying primary pass only lists pixels inside the figure's screen rectangle, the rectangle's columns
    // of a tile row / the pixels of a tile that intersects it (the first nHeavy of a map).
    const size_t tilePixels = static_cast<size_t>(f.tile_size) * f.tile_size;
    p.slotsPerUnit = mapped ? tilePixels : static_cast<size_t>(f.tiles_x) * tilePixels;
    if (!mapped && p.classify && f.rect_valid) {
        const long long rectW = static_cast<long long>(std::min(f.width - 1, f.rect_x1)) - std::max(0, f.rect_x0) + 1;
        p.slotsPerUnit = std::min(p.slotsPerUnit, static_cast<size_t>(std::max<long long>(rectW, 1)) * f.tile_size);
    }
    p.nUnits = mapped ? static_cast<size_t>(spec.nTiles) : static_cast<size_t>(local_tile_rows(f, spec.first, spec.stride));
    p.tilesPerUnit = mapped ? 1 : static_cast<size_t>(f.tiles_x);
    // units that can list pixels at all (the rest need no slots): every row; the heavy tiles of a map
    const size_t nListingUnits = (mapped && p.classify && f.rect_valid) ? static_cast<size_t>(spec.nHeavy) : p.nUnits;
    p.recordBytesPerSlot = static_cast<size_t>(f.spp) * f.draws_per_sample * sizeof(float);
    p.unitsPerChunk = p.nUnits;
    if (p.recordBytesPerSlot > 0 && nListingUnits > 0) {
        const size_t perUnit = p.slotsPerUnit * p.recordBytesPerSlot;
        const size_t fit = std::max<size_t>(1, static_cast<size_t>(ctx.recordBudgetBytes) / std::max<size_t>(1, perUnit));
        // (a map lists its heavy tiles first: chunks of `fit` units hold at most `fit` listing units each)
        if (fit < nListingUnits) p.unitsPerChunk = fit;
    }
    // slot indices are 32-bit
    while (p.unitsPerChunk > 1 && std::min(p.unitsPerChunk, nListingUnits) * p.slotsPerUnit > 0x7fffffffull) --p.unitsPerChunk;
    p.slotCap = std::max<size_t>(1, std::min(p.unitsPerChunk, std::max<size_t>(nListingUnits, 0)) * p.slotsPerUnit);
    p.nChunks = static_cast<int>((p.nUnits + p.unitsPerChunk - 1) / p.unitsPerChunk);
    // Splitting the figure's tiles pays only when the frame (all lanes in flight) has too few tiles to
    // keep every SM busy for as long as its slowest tile takes: below ~10 tiles per SM (B200 sweep:
    // a whole 1080p frame, 2040 tiles, is best unsplit; half a frame is best split in three).
    const long long tilesInFlight = band_tiles(f, spec) * std::max(1, lanesInFlight);
    p.heavyTarget = tilesInFlight * 3 >= 2ll * ctx.smCount * ctx.heavyTilesPerSm
                        ? 0 : ctx.smCount * ctx.heavyTilesPerSm / std::max(1, lanesInFlight);
    p.primaryTarget = ctx.smCount * ctx.primaryBlocksPerSm / std::max(1, lanesInFlight);
    // engine states per tile: one per round of 256 pixels when tiles are split over blocks (kernels.cu)
    p.statesPerTile = static_cast<size_t>(primary_states_per_tile(
        f, static_cast<int>(std::min<size_t>(p.unitsPerChunk * p.tilesPerUnit, 0x7fffffff)), 1, p.primaryTarget, p.heavyTarget));
    // wavefront storage: per path (terminal colour, bounce stack) and per hit-queue entry.  A queue of
    // paths x (bounces + 1) entries cannot overflow; if the budget does not allow it the queue shrinks (to no
    // less than 1.25 entries per path; paths whose hits do not fit are redone in-thread), then the number of
    // paths does (pixels beyond them are shaded by the megakernel).
    if (ctx.shadeMode == 0) {
        const size_t perPath = wavefront_bytes_per_path(f, aov_on(&ctx), aov_guides(ctx.aov), ctx.aov.texel != nullptr), perEntry = wavefront_bytes_per_entry();
        const size_t hitsMax = static_cast<size_t>(wavefront_max_hits_per_path(f));
        const size_t budget = static_cast<size_t>(ctx.waveBudgetBytes);
        const size_t worstPaths = p.slotCap * static_cast<size_t>(f.spp);
        size_t paths = std::min(worstPaths, budget / (perPath + perEntry * std::min<size_t>(hitsMax, 2)));
        paths = std::min<size_t>(paths, 0x7fffff00u);
        paths = std::max<size_t>(paths, static_cast<size_t>(f.spp));
        size_t entries = paths * hitsMax;
        if (ctx.waveQueuePct > 0) entries = std::min(entries, std::max<size_t>(32, paths * static_cast<size_t>(ctx.waveQueuePct) / 100));
        const size_t room = budget > paths * perPath ? (budget - paths * perPath) / perEntry : 0;
        entries = std::min(entries, std::max(room, paths + paths / 4));
        entries = std::min<size_t>(entries, 0xffffff00u);
        p.wavePaths = paths;
        p.waveEntries = entries;
        p.waveBytes = paths * perPath + entries * perEntry + wavefront_fixed_bytes(f) + 16 * 256;
    }
    return p;
}

// Launches the two passes of a band on one stream; output pointers are device memory.  scn: the context whose
// scene (prepared frame, box and texel buffers) is rendered.
int render_bands_lane(McContext* ctx, const McContext* scn, const BandSpec& spec, float4* outF32, uchar4* outU8,
                      cudaStream_t stream, int lanesInFlight = 1) {
    const DevFrame& f = scn->prep.frame;
    const long long nTilesAll = band_tiles(f, spec);
    ctx->chunksLastRender = 0;
    ctx->graphLastRender = false;
    ctx->stats = McRenderStats{};
    ctx->stats.n_samples = static_cast<int64_t>(std::max(f.width, 0)) * std::max(f.height, 0) * f.spp;
    ctx->stats.n_tiles = nTilesAll;
    if (nTilesAll == 0) return MC_OK;
    if (f.width > 65535 || f.height > 65535) return fail(MC_ERR_LIMIT, "image larger than 65535 pixels on a side");
    if (static_cast<long long>(f.tile_size) * f.tile_size > (1ll << 30))
        return fail(MC_ERR_LIMIT, "tile_size too large");
    const BandPlan plan = plan_band(f, spec, *ctx, lanesInFlight);
    if (plan.slotCap > 0x7fffffffull) return fail(MC_ERR_LIMIT, "one tile row holds more than 2^31 pixels");
    const int nChunks = plan.nChunks;

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
    CU_TRY(ctx->slotPixel.reserve(plan.slotCap * sizeof(uint2)));
    CU_TRY(ctx->records.reserve(std::max<size_t>(16, plan.slotCap * plan.recordBytesPerSlot)));
    CU_TRY(ctx->tileStates.reserve(
        std::max<size_t>(16, plan.unitsPerChunk * plan.tilesPerUnit * plan.statesPerTile * 624 * sizeof(uint32_t))));
    CU_TRY(cudaMemsetAsync(ctx->countLog.p, 0, sizeof(unsigned int) * 2 * nChunks, stream));

    while (ctx->passEvents.size() < static_cast<size_t>(3 * nChunks)) {
        cudaEvent_t e;
        CU_TRY(cudaEventCreate(&e));
        ctx->passEvents.push_back(e);
    }
    WaveView wave{};
    const bool aov = aov_on(ctx);
    AovView aovView{};
    aovView.planes = ctx->aov;
    if (ctx->shadeMode == 0) {
        CU_TRY(ctx->wave.reserve(plan.waveBytes));
        if (!wavefront_carve(f, ctx->wave.p, ctx->wave.cap, static_cast<unsigned int>(plan.wavePaths),
                             static_cast<unsigned int>(plan.waveEntries), ctx->smCount * ctx->shadeBlocksPerSm, &wave,
                             aov ? &ctx->aov : nullptr))
            return fail(MC_ERR_CUDA, "wavefront buffer carve failed");
        wave.softGrid = ctx->smCount * ctx->softBlocksPerSm;
        wave.seedMemo = static_cast<uint2*>(scn->seedMemo.p);  // (render_bands has seen to it; the lanes of a frame share it)
        if (!scn->shadowSeedMemo) wave.seedMemo = nullptr;
    }
    if (!ctx->capturing) CU_TRY(cudaEventRecord(ctx->ev0, stream));
    const FramePointers fp = frame_pointers(scn);
    const KernelBuild& build = kernels_for(f);
    const bool mapped = spec.map != nullptr, classify = plan.classify;
    int launches = 0;
    McContext::TileSeedKey seedKey;
    seedKey.width = f.width; seedKey.tile_size = f.tile_size; seedKey.first = spec.first; seedKey.stride = spec.stride;
    seedKey.rows = static_cast<int>(plan.nUnits); seedKey.buf = ctx->tileStates.p; seedKey.stream = stream;
    seedKey.map = spec.map; seedKey.mapVersion = spec.mapVersion;
    seedKey.wordsPerPixel = f.spp * f.draws_per_sample; seedKey.statesPerTile = static_cast<int>(plan.statesPerTile) | (f.rng_mode << 16);
    const bool seedsCacheable = ctx->cacheTileSeeds && nChunks == 1 && f.draws_per_sample > 0;
    const bool seedTiles = !(seedsCacheable && ctx->tileSeedValid && seedKey == ctx->tileSeedKey);
    ctx->tileSeedKey = seedKey;
    ctx->tileSeedValid = false;
    if (seedTiles) ++ctx->seedGen;
    // where the shaded pixels go: this device's memory, or across a link (BandView::far_output)
    const bool farOutput = spec.hotF32 || spec.hotU8 || is_far_memory(ctx, outF32) || is_far_memory(ctx, outU8);
    for (int c = 0; c < nChunks; ++c) {
        const size_t unit0 = static_cast<size_t>(c) * plan.unitsPerChunk;
        const size_t units = std::min<size_t>(plan.unitsPerChunk, plan.nUnits - unit0);
        BandView band{};
        band.out_f32 = outF32;
        band.out_u8 = outU8;
        band.hot_f32 = spec.hotF32;
        band.hot_u8 = spec.hotU8;
        band.far_output = farOutput ? 1 : 0;
        if (ctx->debugPrimaryTiming && nChunks == 1) {  // room for the finest split: one block per 256-pixel round of every tile
            const size_t tilePixels = static_cast<size_t>(f.tile_size) * f.tile_size;
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
            band.first_tile_row = spec.first + static_cast<int>(unit0) * spec.stride;
            band.tile_row_stride = spec.stride;
            band.n_tile_rows = static_cast<int>(units);
            band.out_first_row = spec.outFirst + static_cast<int>(unit0) * spec.outStride;
            band.out_row_stride = spec.outStride;
        }
        ActiveList list;
        list.count = static_cast<unsigned int*>(ctx->countLog.p) + c;
        list.slot_pixel = static_cast<uint2*>(ctx->slotPixel.p);
        list.records = static_cast<float*>(ctx->records.p);
        list.capacity = static_cast<unsigned int>(std::min(plan.slotCap, std::max<size_t>(1, listing * plan.slotsPerUnit)));
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
        const bool seeded = build.launch_primary(f, fp, band, list, classify ? 1 : 0, static_cast<uint32_t*>(ctx->tileStates.p),
                                                 seedTiles, plan.primaryTarget, plan.heavyTarget, stream);
        ctx->tileSeedValid = seedsCacheable && seeded;
        // from here on every pixel of the band outside the figure's screen rectangle is final: the host
        // copy of the image may start (render_host).  Inside a capture this must be a real event-record
        // node, visible to streams outside the graph.
        if (c == nChunks - 1)
            CU_TRY(cudaEventRecordWithFlags(ctx->evPrimaryDone, stream, ctx->capturing ? cudaEventRecordExternal : cudaEventRecordDefault));
        if (!ctx->capturing) CU_TRY(cudaEventRecord(ctx->passEvents[3 * c + 1], stream));
        unsigned int* groupCounter = static_cast<unsigned int*>(ctx->countLog.p) + nChunks + c;
        const int shadeGrid = ctx->smCount * ctx->shadeBlocksPerSm;
        if (ctx->shadeMode == 0)
            build.launch_wavefront(f, fp, band, list, wave, groupCounter, stream, &launches, nullptr, 1, aov ? &aovView : nullptr, nullptr);
        else
            launches += build.launch_shade(f, fp, band, list, shadeGrid, groupCounter, 0u, stream, ctx->shadeMode, &ctx->aov);
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

}  // namespace

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

namespace {

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

void drop_graph(McContext* ctx) {
    if (ctx->graphExec) cudaGraphExecDestroy(ctx->graphExec);
    if (ctx->graph) cudaGraphDestroy(ctx->graph);
    ctx->graphExec = nullptr;
    ctx->graph = nullptr;
}

}  // namespace

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
                 bool frameLayout, const BandSpec* tiles, float4* hotF32, uchar4* hotU8) {
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
        key.aovNormal = ctx->aov.normal; key.aovAlbedo = ctx->aov.albedo; key.aovTexel = ctx->aov.texel;
        if (tiles) {
            key.tileMap = tiles->map; key.mapVersion = tiles->mapVersion; key.nTiles = tiles->nTiles; key.nHeavy = tiles->nHeavy;
        }
        launch_option_bits(ctx, key.optionBits);
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

// Validates a tile list, orders it (tiles the figure's rectangle touches first), uploads it when it changed and
// describes it for render_bands.  *empty: nothing to render.
int prepare_tile_map(McContext* ctx, const int32_t* tiles, int32_t nTiles, cudaStream_t s, BandSpec* spec, bool* empty) {
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

extern "C" {

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

}  // extern "C"
