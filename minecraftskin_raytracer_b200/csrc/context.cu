// context.cu — contexts: creation, options, destruction, the per-device shared contexts, statistics.
#include <cstdlib>
#include "capi_internal.hpp"

// Bumped whenever a device buffer is reallocated: captured frame graphs hold raw pointers.
std::atomic<unsigned long long> g_allocEpoch{1};

namespace {

// One row per option: its name, the environment variable a new context reads it from (or null), the member (an int or
// a long long one), the range a value is clamped to (a range of [0, 1] is a switch: any nonzero value turns it on),
// whether the lanes of a context copy it (inherit_options), and whether it changes what a frame launches (it is then
// part of the key a captured graph is replayed under).
using IntOption = int McOptions::*;
using LongOption = long long McOptions::*;
struct OptionSpec {
    const char* name;
    const char* env;
    IntOption i;
    LongOption ll;
    long long lo, hi;
    bool inherited, launch;
};
constexpr OptionSpec kOptions[] = {
    {"force_all_active", "MCSKIN_FORCE_ALL_ACTIVE", &McOptions::forceAllActive, nullptr, 0, 1, true, true},
    {"record_budget_bytes", nullptr, nullptr, &McOptions::recordBudgetBytes, 1, INT64_MAX, true, true},
    {"shade_blocks_per_sm", "MCSKIN_SHADE_BLOCKS", &McOptions::shadeBlocksPerSm, nullptr, 1, INT32_MAX, true, true},
    {"soft_blocks_per_sm", "MCSKIN_SOFT_BLOCKS", &McOptions::softBlocksPerSm, nullptr, 1, INT32_MAX, true, true},
    {"primary_blocks_per_sm", "MCSKIN_PRIMARY_BLOCKS", &McOptions::primaryBlocksPerSm, nullptr, 0, INT32_MAX, true, true},
    {"heavy_tiles_per_sm", "MCSKIN_HEAVY_TILES", &McOptions::heavyTilesPerSm, nullptr, 0, INT32_MAX, true, true},
    {"batch_lanes", nullptr, &McOptions::batchLanes, nullptr, 1, 16, false, false},
    {"batch_group", "MCSKIN_BATCH_GROUP", &McOptions::batchGroup, nullptr, 1, 4096, false, false},
    {"batch_mode", "MCSKIN_BATCH_MODE", &McOptions::batchMode, nullptr, 0, 1, false, false},
    {"shade_mode", "MCSKIN_SHADE_MODE", &McOptions::shadeMode, nullptr, 0, 2, true, true},
    {"debug_primary_timing", nullptr, &McOptions::debugPrimaryTiming, nullptr, 0, 1, false, true},
    {"wave_queue_pct", "MCSKIN_WAVE_QUEUE_PCT", &McOptions::waveQueuePct, nullptr, 0, 100000, true, true},
    {"frame_lanes", "MCSKIN_FRAME_LANES", &McOptions::frameLanes, nullptr, 1, 8, false, true},
    {"cache_tile_seeds", "MCSKIN_CACHE_TILE_SEEDS", &McOptions::cacheTileSeeds, nullptr, 0, 1, true, true},
    {"use_graphs", "MCSKIN_GRAPHS", &McOptions::useGraphs, nullptr, 0, 1, false, false},
    {"overlap_copy_out", "MCSKIN_OVERLAP_COPY", &McOptions::overlapCopyOut, nullptr, 0, 2, false, false},
    {"wave_budget_bytes", nullptr, nullptr, &McOptions::waveBudgetBytes, 1 << 20, INT64_MAX, true, true},
    {"staged_copy_out", "MCSKIN_STAGED_COPY", &McOptions::stagedCopyOut, nullptr, 0, 1, false, false},
    {"shadow_seed_memo", "MCSKIN_SEED_MEMO", &McOptions::shadowSeedMemo, nullptr, 0, 1, false, true},
};
static_assert(sizeof(kOptions) / sizeof(kOptions[0]) == kOptionCount, "kOptionCount counts the rows of kOptions");

long long option_value(const McOptions& o, const OptionSpec& spec) { return spec.i ? o.*spec.i : o.*spec.ll; }

void set_option_value(McOptions& o, const OptionSpec& spec, long long value) {
    const long long v = spec.lo == 0 && spec.hi == 1 ? value != 0 : std::min(spec.hi, std::max(spec.lo, value));
    if (spec.i) o.*spec.i = static_cast<int>(v);
    else o.*spec.ll = v;
}

}  // namespace

// A lane renders with its parent's options except for the graphs, which the parent captures for all its lanes.
void inherit_options(McContext* lane, const McContext* ctx) {
    for (const OptionSpec& spec : kOptions)
        if (spec.inherited) set_option_value(*lane, spec, option_value(*ctx, spec));
    lane->aov = ctx->aov;
    lane->useGraphs = 0;
}

// The options part of a graph key: the value of every launch option, 0 for the others.
void launch_option_bits(const McContext* ctx, long long* bits) {
    for (size_t i = 0; i < kOptionCount; ++i) bits[i] = kOptions[i].launch ? option_value(*ctx, kOptions[i]) : 0;
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

extern "C" {

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
    for (const OptionSpec& spec : kOptions)
        if (const char* v = spec.env ? std::getenv(spec.env) : nullptr) set_option_value(*ctx, spec, std::atoll(v));
    *out = ctx.release();
    return MC_OK;
}

void mcskin_cuda_context_destroy(McContext* ctx) {
    if (!ctx) return;
    for (McContext* lane : ctx->lanes) mcskin_cuda_context_destroy(lane);
    ctx->lanes.clear();
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (cudaEvent_t e : ctx->pieceEvents) cudaEventDestroy(e);
    ctx->pieceEvents.clear();
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->evCopy) cudaEventDestroy(ctx->evCopy);
    if (ctx->evPrimaryDone) cudaEventDestroy(ctx->evPrimaryDone);
    if (ctx->evFrameDone) cudaEventDestroy(ctx->evFrameDone);
    for (cudaEvent_t e : ctx->evStage)
        if (e) cudaEventDestroy(e);
    if (ctx->copyStream) cudaStreamDestroy(ctx->copyStream);
    if (ctx->evUpload) cudaEventDestroy(ctx->evUpload);
    if (ctx->graphExec) cudaGraphExecDestroy(ctx->graphExec);
    if (ctx->graph) cudaGraphDestroy(ctx->graph);
    for (cudaEvent_t e : ctx->passEvents) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;  // (and with it every buffer)
}

int32_t mcskin_cuda_context_set_option(McContext* ctx, const char* name, int64_t value) {
    if (!ctx || !name) return fail(MC_ERR_INVALID, "set_option: null argument");
    for (const OptionSpec& spec : kOptions) {
        if (std::strcmp(spec.name, name) != 0) continue;
        set_option_value(*ctx, spec, value);
        return MC_OK;
    }
    return fail(MC_ERR_INVALID, std::string("set_option: unknown option ") + name);
}

int32_t mcskin_cuda_context_set_scene(McContext* ctx, const McScene* scene, const McConfig* cfg) {
    if (!ctx || !scene || !cfg) return fail(MC_ERR_INVALID, "set_scene: null argument");
    CU_TRY(cudaSetDevice(ctx->device));
    std::string err;
    const int rc = prepare_frame(scene, cfg, 1, 0.0f, ctx->prep, err);
    if (rc != MC_OK) return fail(rc, err);
    ctx->hasScene = true;
    return upload_scene(ctx);
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

int32_t mcskin_cuda_context_set_aov_targets(McContext* ctx, const McAovTargets* dTargets) {
    if (!ctx) return fail(MC_ERR_INVALID, "set_aov_targets: null context");
    ctx->aov = dTargets ? *dTargets : McAovTargets{};
    return MC_OK;
}

}  // extern "C"
