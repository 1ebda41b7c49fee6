// batch.cu — batches of scenes and skins: grouped launches, frames over the lanes, batches sharded over devices.
#include <cstring>
#include <thread>
#include "capi_internal.hpp"

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
    const size_t waveBytes = (paths * wavefront_bytes_per_path(f0, aov, aov_guides(ctx->aov)) + entries * wavefront_bytes_per_entry() +
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
                                     waveBytes, static_cast<unsigned int>(paths), static_cast<unsigned int>(entries), gridX, &sl.wave, aov ? &av.planes : nullptr))
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
            const KernelBuild& build = kernels_for(f);  // (equal frame descriptions: equal for the whole group)
            // the engines are seeded once per batch — same image geometry for every scene — unless a group is small enough
            // for its tiles to be split over blocks, which changes what is kept per tile
            const int primaryTarget = ctx->smCount * ctx->primaryBlocksPerSm;
            const int statesPerTile = primary_states_per_tile(f, f.tiles_x * f.tiles_y, nS, primaryTarget, 0);
            const bool seedNow = !seeded || statesPerTile != seededStatesPerTile;
            uint32_t* const states = static_cast<uint32_t*>(ctx->tileStates.p);
            // no batched primary kernel for this frame description: frame-by-frame path instead
            if (!build.launch_primary_batch(f, first.band, states, seedNow, gs, nS, first.fp.blob_bytes, primaryTarget, stream)) return MC_OK;
            seeded = true;
            seededStatesPerTile = statesPerTile;
            int launches = 0;
            build.launch_wavefront(f, first.fp, first.band, first.list, first.wave, nullptr, stream, &launches, gs, nS, nullptr, gAov);
        }
        CU_TRY(cudaGetLastError());
    }
    *handled = true;
    return MC_OK;
}

}  // namespace

extern "C" {

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
            DeviceImage img{};
            const int irc = device_image(ctx, outF32, outU8, slots * pixels, &img);
            if (irc != MC_OK) return irc;
            cudaEvent_t copied[2] = {nullptr, nullptr};
            for (auto& e : copied) CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            int rc = MC_OK;
            int half = 0;
            for (size_t c0 = 0; c0 < mine.size() && rc == MC_OK; c0 += chunk, half ^= 1) {
                const int n = static_cast<int>(std::min<size_t>(chunk, mine.size() - c0));
                float4* dF = img.f32 ? img.f32 + static_cast<size_t>(half) * chunk * pixels : nullptr;
                uchar4* dU = img.u8 ? img.u8 + static_cast<size_t>(half) * chunk * pixels : nullptr;
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

}  // extern "C"
