// host_out.cu — frames and tile sets rendered into host images: the copy-out routes and the host-facing render calls.
#include <cstring>
#include "capi_internal.hpp"

namespace {

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

}  // namespace

extern "C" {

// The copy stream waits for the primary pass of every lane of the last render: from then on every pixel outside the
// figure's tiles is final.
static int wait_for_primary_passes(McContext* ctx) {
    CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->evPrimaryDone, 0));
    for (int k = 0; k < ctx->splitLastRender; ++k) CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->lanes[k]->evPrimaryDone, 0));
    return MC_OK;
}

// Waits for the copy stream, the stream and every lane's stream, then checks for errors.
static int finish_frame_streams(McContext* ctx) {
    CU_TRY(cudaStreamSynchronize(ctx->copyStream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    for (McContext* lane : ctx->lanes) CU_TRY(cudaStreamSynchronize(lane->stream));
    CU_TRY(cudaGetLastError());
    return MC_OK;
}

// The pixels of tile columns [tx0, tx1] x rows [ty0, ty1] (hot_tile_range), and the four rectangles of the frame around
// them: above, left, right, below.
static PixelRect tiles_rect(const DevFrame& f, int tx0, int tx1, int ty0, int ty1) {
    const int x0 = tx0 * f.tile_size, y0 = ty0 * f.tile_size;
    return {x0, y0, std::min(f.width, (tx1 + 1) * f.tile_size) - x0, std::min(f.height, (ty1 + 1) * f.tile_size) - y0};
}
static std::vector<PixelRect> frame_outside_tiles(const DevFrame& f, int tx0, int tx1, int ty0, int ty1) {
    const PixelRect t = tiles_rect(f, tx0, tx1, ty0, ty1);
    const int x1 = t.x + t.w, y1 = t.y + t.h;
    return {{0, 0, f.width, t.y}, {0, t.y, t.x, t.h}, {x1, t.y, f.width - x1, t.h}, {0, y1, f.width, f.height - y1}};
}

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
    const bool dual = mappedHost && ctx->overlapCopyOut >= 2 && classified && !ctx->tileMapLightRects.empty();
    if (mappedHost && !dual)  // every tile straight into the host image
        return render_bands(ctx, 0, 1, static_cast<float4*>(aliasF32), static_cast<uchar4*>(aliasU8), ctx->stream, true, &spec);
    DeviceImage img{};
    rc = device_image(ctx, hostF32, hostU8, static_cast<size_t>(f.width) * f.height, &img);
    if (rc != MC_OK) return rc;
    if (!dual) {
        rc = render_bands(ctx, 0, 1, img.f32, img.u8, ctx->stream, true, &spec);
        if (rc != MC_OK) return rc;
        return copy_rects_to_host(tile_rects(f, ctx->tileMapOrdered), f.width, img.f32, hostF32, img.u8, hostU8, ctx->stream);
    }
    rc = render_bands(ctx, 0, 1, img.f32, img.u8, ctx->stream, true, &spec, static_cast<float4*>(aliasF32),
                      static_cast<uchar4*>(aliasU8));
    if (rc != MC_OK) return rc;
    rc = wait_for_primary_passes(ctx);
    if (rc != MC_OK) return rc;
    return copy_rects_to_host(ctx->tileMapLightRects, f.width, img.f32, hostF32, img.u8, hostU8, ctx->copyStream);
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
    rc = finish_frame_streams(ctx);
    if (rc != MC_OK) return rc;
    if (msDevice && nTiles > 0) CU_TRY(cudaEventElapsedTime(msDevice, ctx->ev0, ctx->ev1));
    return MC_OK;
}

// A whole frame into PAGEABLE host images (an Image's std::vector<Color>, a numpy array): the dual-destination route
// of render_host with the library's own page-locked staging images in the caller's place, and host threads that move
// every piece on to the caller's memory as soon as it has arrived — the 93 % of a frame that are final after the primary
// pass cross PCIe and the host's memory while the GPU shades; only the figure's tiles are left when the last kernel ends.
// (One copy of the whole image from device memory followed by one memcpy, the route without this, takes ~4 ms at 1080p.)
static int render_host_staged(McContext* ctx, const DeviceImage& img, float* outF32, uint8_t* outU8, int tx0, int tx1, int ty0,
                              int ty1, McRenderStats* stats) {
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
    int rc = render_bands(ctx, 0, 1, img.f32, img.u8, ctx->stream, false, nullptr, static_cast<float4*>(aliasF32),
                          static_cast<uchar4*>(aliasU8));
    if (rc != MC_OK) return rc;
    rc = wait_for_primary_passes(ctx);
    if (rc != MC_OK) return rc;
    const int W = f.width;
    // pieces of about 2 MB of float pixels: whole rows of the four rectangles around the figure's tiles, then of those tiles
    std::vector<PixelRect> light, hot;
    auto cut = [&](std::vector<PixelRect>& into, const PixelRect& r) {
        if (r.w <= 0 || r.h <= 0) return;
        const int rowsPerPiece = std::max(1, (2 << 20) / (r.w * 16));
        for (int y = 0; y < r.h; y += rowsPerPiece) into.push_back({r.x, r.y + y, r.w, std::min(rowsPerPiece, r.h - y)});
    };
    for (const PixelRect& r : frame_outside_tiles(f, tx0, tx1, ty0, ty1)) cut(light, r);
    cut(hot, tiles_rect(f, tx0, tx1, ty0, ty1));
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
        rc = copy_rects_to_host({light[i]}, W, img.f32, outF32 ? static_cast<float*>(ctx->stageF32.p) : nullptr, img.u8,
                                outU8 ? static_cast<uint8_t*>(ctx->stageU8.p) : nullptr, ctx->copyStream);
        if (rc != MC_OK) return rc;
        CU_TRY(cudaEventRecord(ctx->pieceEvents[i], ctx->copyStream));
        add_jobs(light[i], ctx->pieceEvents[i]);
    }
    if (!run_host_copies(ctx->device, jobs)) CU_TRY(cudaGetLastError());
    rc = finish_frame_streams(ctx);
    if (rc != MC_OK) return rc;
    jobs.clear();
    for (const PixelRect& r : hot) add_jobs(r, nullptr);
    run_host_copies(ctx->device, jobs);
    return finish_stats(ctx, stats);
}

// A whole frame rendered into host images (either may be null).
static int render_host(McContext* ctx, const McScene* scene, const McConfig* cfg, float* outF32, uint8_t* outU8, McRenderStats* stats) {
    int rc = mcskin_cuda_context_set_scene(ctx, scene, cfg);
    if (rc != MC_OK) return rc;
    const DevFrame& f = ctx->prep.frame;
    const size_t pixels = static_cast<size_t>(f.width) * f.height;
    DeviceImage img{};
    rc = device_image(ctx, outF32, outU8, pixels, &img);
    if (rc != MC_OK) return rc;
    // Two destinations (whole frames into page-locked images the device can address): the tiles the figure's screen
    // rectangle touches — the only ones with pixels that are final as late as the frame's last kernel — are written by
    // the kernels straight into the caller's image (a few MB over PCIe, spread over the frame); all other tiles are
    // final after the primary passes and leave the device image by DMA then, next to the shading kernels.  Nothing
    // is left to copy when the last kernel ends.
    int tx0 = 0, tx1 = -1, ty0 = 0, ty1 = -1;
    const bool classified = !ctx->forceAllActive && f.spp <= kBlockThreads;
    void* aliasF32 = (ctx->overlapCopyOut && classified && outF32) ? device_alias_of_host(outF32) : nullptr;
    void* aliasU8 = (ctx->overlapCopyOut && classified && outU8) ? device_alias_of_host(outU8) : nullptr;
    const bool dual = ctx->overlapCopyOut >= 2 && classified && hot_tile_range(f, &tx0, &tx1, &ty0, &ty1) &&
                      (!outF32 || aliasF32) && (!outU8 || aliasU8);
    if (!dual && ctx->stagedCopyOut && ctx->overlapCopyOut >= 2 && classified && (outF32 || outU8) &&
        !(outF32 && is_pinned_host(outF32)) && !(outU8 && is_pinned_host(outU8)) && hot_tile_range(f, &tx0, &tx1, &ty0, &ty1)) {
        rc = render_host_staged(ctx, img, outF32, outU8, tx0, tx1, ty0, ty1, stats);
        if (rc != MC_ERR_LIMIT) return rc;
    }
    if (dual) {
        rc = render_bands(ctx, 0, 1, img.f32, img.u8, ctx->stream, false, nullptr, static_cast<float4*>(aliasF32),
                          static_cast<uchar4*>(aliasU8));
        if (rc != MC_OK) return rc;
        rc = wait_for_primary_passes(ctx);
        if (rc != MC_OK) return rc;
        rc = copy_rects_to_host(frame_outside_tiles(f, tx0, tx1, ty0, ty1), f.width, img.f32, outF32, img.u8, outU8, ctx->copyStream);
        if (rc != MC_OK) return rc;
        rc = finish_frame_streams(ctx);
        if (rc != MC_OK) return rc;
        return finish_stats(ctx, stats);
    }
    rc = render_bands(ctx, 0, 1, img.f32, img.u8, ctx->stream);
    if (rc != MC_OK) return rc;
    // Copy-out overlapped with shading: once the primary passes are done, every pixel outside the
    // figure's screen rectangle is final (93 % of the headline frame), so the whole image starts its
    // way to the host then, next to the shading kernels; when the frame is complete only the
    // rectangle is sent again.  Needs page-locked destinations (DMA straight into the caller's
    // buffers) and a whole frame in one chunk.
    // (and the classifying primary pass: without it every pixel is written by the shading pass)
    const bool overlap = ctx->overlapCopyOut && f.rect_valid && ctx->chunksLastRender == 1 &&
                         !ctx->forceAllActive && f.spp <= kBlockThreads && f.rect_x0 <= f.rect_x1 && f.rect_y0 <= f.rect_y1 &&
                         (!outF32 || is_pinned_host(outF32)) && (!outU8 || is_pinned_host(outU8));
    if (overlap) {
        rc = wait_for_primary_passes(ctx);
        if (rc != MC_OK) return rc;
        if (outF32) CU_TRY(cudaMemcpyAsync(outF32, img.f32, pixels * sizeof(float4), cudaMemcpyDeviceToHost, ctx->copyStream));
        if (outU8) CU_TRY(cudaMemcpyAsync(outU8, img.u8, pixels * sizeof(uchar4), cudaMemcpyDeviceToHost, ctx->copyStream));
        CU_TRY(cudaEventRecord(ctx->evFrameDone, ctx->stream));
        CU_TRY(cudaStreamWaitEvent(ctx->copyStream, ctx->evFrameDone, 0));
        const int x0 = std::max(0, f.rect_x0), x1 = std::min(f.width - 1, f.rect_x1);
        const int y0 = std::max(0, f.rect_y0), y1 = std::min(f.height - 1, f.rect_y1);
        rc = copy_rects_to_host({{x0, y0, x1 - x0 + 1, y1 - y0 + 1}}, f.width, img.f32, outF32, img.u8, outU8, ctx->copyStream);
        if (rc != MC_OK) return rc;
        CU_TRY(cudaStreamSynchronize(ctx->copyStream));
    } else {
        if (outF32) {
            rc = copy_out(ctx, outF32, img.f32, pixels * sizeof(float4));
            if (rc != MC_OK) return rc;
        }
        if (outU8) {
            rc = copy_out(ctx, outU8, img.u8, pixels * sizeof(uchar4));
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
    rc = render_host(ctx, scene, cfg, outF32, outU8, stats);
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
        if (want.normal) std::fill(want.normal, want.normal + 3 * pixels, 0.0f);
        if (want.albedo) std::fill(want.albedo, want.albedo + 4 * pixels, 0.0f);
        if (stats) *stats = McRenderStats{};
        return MC_OK;
    }
    std::lock_guard<std::mutex> lock(g_ctxMutex);
    McContext* ctx = nullptr;
    int rc = shared_context(device, &ctx);
    if (rc != MC_OK) return rc;
    CU_TRY(cudaSetDevice(ctx->device));
    CU_TRY(ctx->aovPlanes.reserve(std::max<size_t>(16, pixels * 10 * sizeof(float))));  // 1 + 1 + 1 + 3 + 4 values a pixel
    float* const base = static_cast<float*>(ctx->aovPlanes.p);
    McAovTargets dev{};
    dev.coverage = want.coverage ? base : nullptr;
    dev.depth = want.depth ? base + pixels : nullptr;
    dev.tri_id = want.tri_id ? reinterpret_cast<int32_t*>(base + 2 * pixels) : nullptr;
    dev.normal = want.normal ? base + 3 * pixels : nullptr;
    dev.albedo = want.albedo ? base + 6 * pixels : nullptr;
    ctx->aov = dev;
    rc = render_host(ctx, scene, cfg, outF32, outU8, stats);
    ctx->aov = McAovTargets{};
    if (rc != MC_OK) return rc;
    // (render_host has synchronised with the frame)
    if (want.coverage) CU_TRY(cudaMemcpyAsync(want.coverage, dev.coverage, pixels * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (want.depth) CU_TRY(cudaMemcpyAsync(want.depth, dev.depth, pixels * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (want.tri_id) CU_TRY(cudaMemcpyAsync(want.tri_id, dev.tri_id, pixels * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (want.normal) CU_TRY(cudaMemcpyAsync(want.normal, dev.normal, 3 * pixels * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (want.albedo) CU_TRY(cudaMemcpyAsync(want.albedo, dev.albedo, 4 * pixels * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(cudaStreamSynchronize(ctx->stream));
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
    DeviceImage img{};
    rc = device_image(ctx, true, true, pixels, &img);
    if (rc != MC_OK) return rc;
    // render the whole tile row (cheap) and copy back only the tile's columns
    rc = render_bands(ctx, tileRow, f.tiles_y, img.f32, img.u8, ctx->stream);
    if (rc != MC_OK) return rc;
    CU_TRY(cudaStreamSynchronize(ctx->stream));
    if (imageF32)
        CU_TRY(cudaMemcpy2D(imageF32 + (static_cast<size_t>(tile->y) * f.width + tile->x) * 4, f.width * sizeof(float4),
                            img.f32 + tile->x, f.width * sizeof(float4),
                            tile->width * sizeof(float4), tile->height, cudaMemcpyDeviceToHost));
    if (imageU8)
        CU_TRY(cudaMemcpy2D(imageU8 + (static_cast<size_t>(tile->y) * f.width + tile->x) * 4, f.width * sizeof(uchar4),
                            img.u8 + tile->x, f.width * sizeof(uchar4),
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
        CU_TRY(cudaSetDevice(ctxs[d]->device));
        int rc = finish_frame_streams(ctxs[d]);
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

}  // extern "C"
