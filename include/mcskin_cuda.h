/*
 * mcskin_cuda.h — C ABI of the B200-native render hot path.
 *
 * This is the drop-in boundary for MCSkin RaytraceRenderer's
 *     Image TileRenderer::render(const Scene&, const RayTracer::Config&, progress)
 * (reference: src/raytracer/tile_renderer.h:26-28, tile_renderer.cpp:129-189).
 * The reference has no FFI of its own (it is one C++ process); the C++ wrapper in
 * include/mcskin/raytracer/tile_renderer.h keeps the reference's signature and
 * flattens Scene/Config into the PODs below before calling these entry points.
 * INTEGRATION.md shows the binding a maintainer adds on the reference side.
 *
 * Rules of the ABI: plain pointers and sizes, fixed-width PODs, no STL, no torch
 * types, no exceptions.  Every function returns 0 on success or a negative
 * MC_ERR_* code; mcskin_cuda_last_error() returns the thread-local message.
 * There is no CPU fallback: without a CUDA device every compute call fails with
 * MC_ERR_NO_DEVICE.
 */
#ifndef MCSKIN_CUDA_H
#define MCSKIN_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCSKIN_ABI_VERSION 4

enum {
    MC_OK = 0,
    MC_ERR_INVALID = -1,   /* bad argument (null pointer, negative size, bad texture window) */
    MC_ERR_NO_DEVICE = -2, /* no CUDA device / driver */
    MC_ERR_CUDA = -3,      /* a CUDA runtime call or kernel failed */
    MC_ERR_LIMIT = -4      /* scene exceeds a documented limit */
};

/* One face texture = a window of `width*height` RGBA float texels in the scene's
 * texel pool (row-major).  Mirrors TextureRegion (src/skin/texture_region.h:7-27).
 *   texel_offset <  0              : null Triangle::texture  -> opaque magenta (intersection.cpp:303-306)
 *   width <= 0 || height <= 0      : empty region            -> (0,0,0,1)      (texture_region.h:20-22) */
typedef struct McFaceTex {
    int32_t texel_offset;
    int32_t width;
    int32_t height;
} McFaceTex;

/* One Mesh, which the reference intersects as ONE axis-aligned box
 * (src/raytracer/intersection.cpp:200-406, src/scene/mesh.h:12-30).
 * bounds_* are the min/max over the vertices of the triangle list the reference
 * uses for that mesh: Mesh::localTriangles when has_rotation, else Mesh::triangles
 * (intersection.cpp:45-64,374-395).  face[f] is the texture of
 * Mesh::triangles[2*f] for the reference face index f = 0..5
 * (-Z,+Z,+X,-X,+Y,-Y; intersection.cpp:86-129). */
typedef struct McBox {
    float bounds_min[3];
    float bounds_max[3];
    float pivot[3];        /* Mesh::pivot */
    float rot_x_deg;       /* Mesh::rotX */
    float rot_z_deg;       /* Mesh::rotZ */
    int32_t has_rotation;  /* Mesh::hasRotation */
    int32_t is_outer_layer;/* Mesh::isOuterLayer */
    int32_t n_triangles;   /* size of the list the bounds came from; 0 -> never hit (intersection.cpp:205) */
    McFaceTex face[6];
} McBox;

/* Scene (src/scene/scene.h:10-34).  Light::intensity is never read by the
 * reference and is not carried. */
typedef struct McScene {
    int32_t n_boxes;
    const McBox* boxes;
    int32_t n_texels;
    const float* texels_rgba; /* n_texels * 4 floats */
    float light_pos[3];
    float light_color[4];
    float light_radius;
    float cam_pos[3];
    float cam_target[3];
    float cam_up[3];
    float cam_fov_deg;
    float background[4];
} McScene;

/* RayTracer::Config (src/raytracer/raytracer.h:10-38) + ShadingParams
 * (src/raytracer/shading.h:9-14).  thread_count is accepted and ignored. */
typedef struct McConfig {
    int32_t width, height;
    int32_t max_bounces;
    int32_t samples_per_pixel;
    int32_t tile_size;
    int32_t thread_count;
    int32_t soft_shadows;
    int32_t shadow_samples;
    int32_t ao_enabled;
    int32_t ao_samples;
    float ao_radius;
    float ao_intensity;
    int32_t dof_enabled;
    float aperture;
    float focus_distance;
    int32_t gradient_bg;
    float gradient_scale;
    float bg_center[4];
    float bg_edge[4];
    float kd, ks, ambient, shininess;
    /* Not in the reference's Config.  0: every random stream is the reference's std::mt19937 (frames equal the
     * reference's bit for bit).  1 (MC_RNG_COUNTER): counter-based streams — draw k of a stream seeded s is
     * canonical(mc_rng_counter_word(s, k)), no engine state, no 623-step seeding per tile and per shaded hit; the
     * same seeds, the same number and order of draws, the same float mapping.  Frames then differ from the
     * reference's in their noise only and equal the CPU oracle's with the same switch. */
    int32_t rng_mode;
} McConfig;
#define MC_RNG_MT19937 0
#define MC_RNG_COUNTER 1

/* Word k of the counter-based stream seeded `seed` (rng_mode 1): two rounds of the lowbias32 integer hash. */
static inline uint32_t mc_rng_lowbias32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
static inline uint32_t mc_rng_counter_key(uint32_t seed) { return mc_rng_lowbias32(seed ^ 0x9e3779b9u); }
static inline uint32_t mc_rng_counter_word(uint32_t seed, uint32_t k) { return mc_rng_lowbias32(mc_rng_counter_key(seed) + k); }
/* The same word from the library (for bindings that restate the hash in their own language and want to check it). */
uint32_t mcskin_counter_word(uint32_t seed, uint32_t k);

/* Fills *cfg with the reference defaults (raytracer.h:10-38, shading.h:9-14). */
void mcskin_config_defaults(McConfig* cfg);

/* Tile = {x, y, width, height} (tile_renderer.h:11-14). */
typedef struct McTile {
    int32_t x, y, width, height;
} McTile;

/* TileRenderer::generateTiles (tile_renderer.cpp:18-39).  Returns the tile count
 * (0 for non-positive arguments); writes at most `capacity` tiles when out != NULL. */
int32_t mcskin_generate_tiles(int32_t image_width, int32_t image_height, int32_t tile_size,
                              McTile* out, int32_t capacity);

/* progress(done, total, user): called on the calling thread, exactly `total`
 * (= tile count) times with done = 1..total (tile_renderer.cpp:168-172). */
typedef void (*McProgressFn)(int32_t done, int32_t total, void* user);

/* Per-frame counters written by the device (all optional). */
typedef struct McRenderStats {
    int32_t n_tiles;
    int32_t n_active_pixels;   /* pixels with at least one primary sample hitting geometry */
    int64_t n_samples;         /* width*height*spp */
    float ms_device;           /* CUDA-event time of the kernels of this call */
    int32_t n_kernel_launches; /* kernels launched by this call */
    float ms_primary;          /* of which: primary (classification + background) pass */
    float ms_shade;            /* of which: shading pass */
} McRenderStats;

int32_t mcskin_cuda_device_count(void);
const char* mcskin_cuda_last_error(void);
int32_t mcskin_cuda_abi_version(void);
/* sizeof of McFaceTex, McBox, McScene, McConfig, McTile, McRenderStats, McRay, McHit
 * as compiled, so a binding can verify its mirror of this header. */
void mcskin_cuda_abi_sizes(int32_t* out8);

/* TileRenderer::render (tile_renderer.h:26-28, tile_renderer.cpp:129-189): host scene in, host image out
 * (row-major, width*height pixels).  With page-locked destinations the image leaves for the host while the
 * shading pass still runs.
 * out_rgba_f32 : width*height*4 floats (Image::pixels), may be NULL
 * out_rgba_u8  : width*height*4 bytes, uint8(clamp(c)*255+0.5) (image_writer.cpp:18-22), may be NULL
 * Renders on the current thread's CUDA device `device` (>= 0).
 * Some configurations make NaN channels in the reference (ao_samples == 0 with AO on: 0/0 in computeAO; a negative
 * shininess: inf*0 in shade()).  They are stored as x86's default NaN 0xffc00000, the bits the reference writes, here
 * and in the float outputs of the single-query calls below (trace, shade, ambient_occlusion); their 8-bit value is 0.
 * NaN payloads carried in by the inputs (NaN texels or config values) are not reproduced. */
int32_t mcskin_cuda_render(const McScene* scene, const McConfig* cfg, int32_t device,
                           float* out_rgba_f32, uint8_t* out_rgba_u8,
                           McProgressFn progress, void* user, McRenderStats* stats);

/* Per-pixel planes rendered in the same pass as the colour ("AOVs"), each width*height values indexed like the colour
 * image of the same call; any member may be NULL.  For pixel (px, py) with samples s = 0..spp-1 in the renderer's sample
 * order, let h_s be the closest hit of sample s's camera ray exactly as the colour pass builds it (jitter, thin lens,
 * either rng_mode; the query whose miss gives the sample the gradient, tile_renderer.cpp:111), and n the number of
 * samples that hit.  Independent of max_bounces, shading, shadows and AO:
 *   coverage : (float)n * (1.0f / (float)spp)
 *   depth    : the hit distances h_s.t of the hitting samples summed left to right from 0.0f, divided by (float)n;
 *              0.0f when n == 0
 *   tri_id   : box*12 + face*2 of the first hitting sample (the McHit / mcskin_cuda_aov convention); -1 when n == 0
 * The guide planes a denoiser or compositor takes next to the colour, 3 and 4 floats per pixel (pixel i at 3*i, 4*i):
 *   normal   : McHit.normal of the hitting samples (the outer-layer exit-face flip included, posed boxes back-transformed),
 *              each component summed left to right from 0.0f (so a -0 component reads +0) and divided by (float)n; not
 *              renormalised.  (0, 0, 0) when n == 0
 *   albedo   : the same fold over McHit.tex_color (magenta for a null texture, (0, 0, 0, 1) for an empty region);
 *              (0, 0, 0, 0) when n == 0
 * A hit never has a texel of alpha 0: such texels are passed through, and the outer-layer exit face is taken only when
 * its alpha is > 0.  So when no texel alpha is negative (every skin built from an 8-bit atlas), albedo's alpha is > 0
 * exactly where tri_id >= 0.
 * The skin-texel plane, one int32 per pixel: which texel of the scene's texture the pixel shows.
 *   texel    : the texel index the first hitting sample's closest hit took (the sample tri_id reports), into
 *              scene.texels_rgba: texels_rgba[4*texel .. 4*texel+3] == McHit.tex_color of that hit (for an outer-layer
 *              hit that fell through to the exit face, the exit face's texel).  A face without texels gives the index
 *              of a synthetic texel just past the pool: n_texels for a null texture (McFaceTex.texel_offset < 0,
 *              magenta) and n_texels + 1 for an empty region (width <= 0 or height <= 0, (0, 0, 0, 1)).  -1 when n == 0,
 *              so texel >= 0 exactly where tri_id >= 0.  In image i of a batch it indexes scene i's texels.
 * (normal and albedo were appended in ABI version 3, texel in ABI version 4.) */
typedef struct McAovTargets {
    float* coverage;
    float* depth;
    int32_t* tri_id;
    float* normal;
    float* albedo;
    int32_t* texel;
} McAovTargets;

/* mcskin_cuda_render with AOV planes: the same colour bytes, and the planes `aov` asks for (host memory, width*height
 * values each, 3 and 4 times that for normal and albedo; aov may be NULL).  A frame with no tiles leaves the defaults
 * (0, 0, -1, zeros, zeros, -1) in every requested plane. */
int32_t mcskin_cuda_render_aovs(const McScene* scene, const McConfig* cfg, int32_t device,
                                float* out_rgba_f32, uint8_t* out_rgba_u8, const McAovTargets* aov,
                                McRenderStats* stats);

/* TileRenderer::renderTile (tile_renderer.cpp:71-127): renders one tile into the
 * caller's full-size image buffers (only the tile's pixels are written). */
int32_t mcskin_cuda_render_tile(const McScene* scene, const McConfig* cfg, int32_t device,
                                const McTile* tile, float* image_rgba_f32, uint8_t* image_rgba_u8);

/* Same frame split over devices 0..n_devices-1 of this process: every device renders its cost-balanced tile set
 * (mcskin_partition_tiles) and sends it to the caller's image over its own PCIe link (page-locked, mapped images:
 * see mcskin_cuda_context_render_scene_tiles). */
int32_t mcskin_cuda_render_multi(const McScene* scene, const McConfig* cfg, int32_t n_devices,
                                 float* out_rgba_f32, uint8_t* out_rgba_u8, McRenderStats* stats);

/* ---- device-resident interface (bench `value`, torch.distributed band gather) ---- */
typedef struct McContext McContext;

int32_t mcskin_cuda_context_create(int32_t device, McContext** out);
void mcskin_cuda_context_destroy(McContext* ctx);
/* Uploads and pre-processes scene+config (host trig, camera basis, texel pool). */
int32_t mcskin_cuda_context_set_scene(McContext* ctx, const McScene* scene, const McConfig* cfg);
/* Renders tile rows {first_tile_row + k*tile_row_stride} into device buffers laid
 * out as a compact band image: the local tile rows in increasing order, each
 * tile_size pixel rows (last one clipped), width*4 channels per row.
 * d_out_f32 / d_out_u8 are DEVICE pointers (either may be 0).  stream is a
 * cudaStream_t passed as void* (0 = default stream).  Asynchronous. */
int32_t mcskin_cuda_context_render_bands(McContext* ctx, int32_t first_tile_row, int32_t tile_row_stride,
                                         void* d_out_f32, void* d_out_u8, void* stream);
/* Number of pixel rows the call above writes for that partition. */
int32_t mcskin_cuda_band_rows(const McConfig* cfg, int32_t first_tile_row, int32_t tile_row_stride);
/* The same rows written at their own place in a FULL-frame image (width*height pixels, rows in
 * image order) instead of a compact band.  The image may live on another device of the box: with
 * peer access (see mcskin_cuda_ipc_open) every GPU stores its tile rows straight into the root's
 * frame over NVLink and no gather step is left — only a barrier before the root reads it. */
int32_t mcskin_cuda_context_render_rows_into_frame(McContext* ctx, int32_t first_tile_row, int32_t stride,
                                                    void* d_frame_f32, void* d_frame_u8, void* stream);
/* Any set of whole tiles (frame tile indices ty*tiles_x + tx, each at most once, any order) written at their
 * own place in a FULL-frame image — the unit the reference's own load balancer hands out
 * (tile_renderer.cpp:148-186: threads steal tiles from an atomic counter).  Every tile has its own jitter stream
 * (tile_renderer.cpp:78), so any partition of a frame into tile sets gives the bits of the whole frame.  With
 * mcskin_partition_tiles this is the multi-GPU split of one frame: cost-balanced tile sets, stored by every GPU
 * straight into the root's frame (peer memory) or into one page-locked host frame (mcskin_cuda_host_register). */
int32_t mcskin_cuda_context_render_tiles_into_frame(McContext* ctx, const int32_t* tiles, int32_t n_tiles,
                                                     void* d_frame_f32, void* d_frame_u8, void* stream);
/* The per-frame call of a rank whose scene lives on the CPU and whose result goes to a HOST image shared by every rank
 * of the box: set_scene (upload) + this rank's tiles + wait.  host_frame_* must be page-locked and mapped
 * (mcskin_cuda_host_register, cudaHostAlloc, torch pin_memory).  The tiles the figure's screen rectangle touches are
 * stored by the kernels straight into the host image; the others are final after the primary pass and leave a
 * device image by DMA, as a few rectangles, next to the shading kernels.  *ms_device (may be null): the frame's
 * kernels, CUDA events.  Blocking. */
int32_t mcskin_cuda_context_render_scene_tiles(McContext* ctx, const McScene* scene, const McConfig* cfg,
                                                const int32_t* tiles, int32_t n_tiles, float* host_frame_f32,
                                                uint8_t* host_frame_u8, float* ms_device);
/* Deals the tiles of a frame to n_parts renderers so that every part costs about the same: tiles are weighted
 * by how much of them the figure's screen rectangles cover (covered pixels cost ~50x a background pixel) and
 * dealt greedily, heaviest first, to the least loaded part; the background tiles are then dealt as contiguous runs
 * in frame order that fill every part to the same level (a part's background is a few rectangles); deterministic, the
 * parts are disjoint and cover the frame.  root_part: the part whose device holds the frame the others store into over
 * NVLink (their background tiles count 1.3: remote stores), or -1 when every part writes under the same conditions.  Returns the number of tiles of `part` (negative MC_ERR_* on failure) and writes at most `capacity`
 * of them to out_tiles (may be null to query the count).  Host code only: needs no device. */
int32_t mcskin_partition_tiles(const McScene* scene, const McConfig* cfg, int32_t n_parts, int32_t part,
                               int32_t root_part, int32_t* out_tiles, int32_t capacity);
/* Host code only: copies `rows` rows of `row_bytes` from src to dst (pitches in bytes), cut into `pieces` jobs for the
 * library's host copy threads — the ones that carry a frame from the page-locked staging image into a pageable
 * destination (mcskin_cuda_render into an Image's std::vector<Color>) while the GPU is still shading.  Needs no device. */
int32_t mcskin_host_copy_rows(void* dst, const void* src, uint64_t dst_pitch, uint64_t src_pitch, uint64_t row_bytes,
                              uint64_t rows, int32_t pieces);
/* Page-locks a host range (e.g. a shared-memory segment every process of the box has mapped) and maps it into
 * the device address space: *d_ptr is what kernels store to (zero-copy over PCIe), so N GPUs can write their
 * tiles of one frame into one host image through N PCIe links at once. */
int32_t mcskin_cuda_host_register(void* host_ptr, uint64_t bytes, void** d_ptr);
int32_t mcskin_cuda_host_unregister(void* host_ptr);
/* Plain device allocations that can be shared between the processes of one box (one process per
 * GPU): export on the owner, open on the peers (cudaIpcGetMemHandle / cudaIpcOpenMemHandle; the
 * handle is 64 opaque bytes to pass over any channel, e.g. a torch.distributed broadcast). */
int32_t mcskin_cuda_device_alloc(int32_t device, uint64_t bytes, void** out_ptr);
int32_t mcskin_cuda_device_free(int32_t device, void* ptr);
int32_t mcskin_cuda_ipc_export(int32_t device, void* ptr, uint8_t handle_out[64]);
int32_t mcskin_cuda_ipc_open(int32_t device, const uint8_t handle[64], void** out_ptr);
int32_t mcskin_cuda_ipc_close(int32_t device, void* ptr);
/* Stream-ordered flags in (peer-mapped) device memory, the barrier of the peer-store exchange:
 * signal stores `value` into *d_flag with system-scope release semantics after everything queued
 * before it on `stream` (so a peer that sees the value also sees the rows stored before it);
 * wait holds `stream` until each of the n 32-bit flags is >= value (acquire), or ~2 s have passed
 * (then *d_timeout, if given, is set to 1 and the stream continues: no device hang on a dead peer). */
int32_t mcskin_cuda_peer_signal(int32_t device, void* d_flag, uint32_t value, void* stream);
/* One process driving several devices: lets kernels on `device` address memory allocated on `peer` (frames opened
 * with mcskin_cuda_ipc_open need no such call). */
int32_t mcskin_cuda_enable_peer_access(int32_t device, int32_t peer);
int32_t mcskin_cuda_peer_wait(int32_t device, const void* d_flags, int32_t n, uint32_t value, void* d_timeout, void* stream);
/* Diagnosis: with the option "debug_primary_timing" (one lane, no graph) the blocks of the pixel-per-lane primary
 * kernels record when they ran: 4 words per block (entry ns, exit ns, frame tile, part | parts << 16; zeros for
 * blocks that had nothing to do).  Returns the number of records of the last launch. */
int32_t mcskin_cuda_context_debug_block_times(McContext* ctx, uint64_t* out, int32_t capacity);
/* AOV planes for the context's later render calls: d_targets holds DEVICE-addressable pointers (copied; NULL, or all
 * members NULL, switches the planes off).  render_bands, render_rows_into_frame, render_tiles_into_frame, render_batch and
 * render_skin_batch then write every plane that is set for every pixel they render, at the colour image's index (image i
 * of a batch at offset i*width*height, times 3 for normal and 4 for albedo); frame lanes inherit the targets.  render_scene_tiles fails with MC_ERR_INVALID
 * while targets are set. */
int32_t mcskin_cuda_context_set_aov_targets(McContext* ctx, const McAovTargets* d_targets);
/* Blocks until the context's work is done, fills stats of the last render. */
int32_t mcskin_cuda_context_sync(McContext* ctx, McRenderStats* stats);
/* Tuning / test knobs (every combination renders the same bits; INTEGRATION.md §6 has the table):
 * "frame_lanes" (streams a frame's tile rows are dealt to), "use_graphs" (replay a repeated frame as a CUDA
 * graph), "cache_tile_seeds", "wave_queue_pct" (hit-queue entries as a percentage of the paths; 0 = cannot overflow),
 * "soft_blocks_per_sm", "wave_budget_bytes",
 * "record_budget_bytes", "shade_blocks_per_sm", "primary_blocks_per_sm", "heavy_tiles_per_sm",
 * "shade_mode" (0 wavefront, 1/2 megakernel forms), "force_all_active" (0/1: skip the hit/miss
 * classification and shade every pixel), "overlap_copy_out", "batch_mode", "batch_group", "batch_lanes".
 * Unknown names return MC_ERR_INVALID. */
int32_t mcskin_cuda_context_set_option(McContext* ctx, const char* name, int64_t value);

/* Batched renders (one skin per scene, same config), scene i -> image i (SURVEY.md §8e).
 * d_out_* are device pointers to n_scenes consecutive images.  Asynchronous.  Scenes that share a frame
 * description (image size, sampling, camera, light, box layout) are rendered by one set of launches whose
 * gridDim.y is the scene, "batch_group" scenes at a time; with "batch_mode" 0, or for frame descriptions
 * without a batched kernel form, frames are pipelined one by one over "batch_lanes" internal streams.
 * The given stream (or the context's) carries or waits for all of it; mcskin_cuda_context_sync blocks
 * until the images are complete. */
int32_t mcskin_cuda_context_render_batch(McContext* ctx, const McScene* scenes, int32_t n_scenes,
                                         const McConfig* cfg, void* d_out_f32, void* d_out_u8, void* stream);
/* The flat scene of a skin WITHOUT its float texels (host code): the boxes mcskin_build_skin_scene would emit, their
 * face windows into a texel pool of scene_out->n_texels texels that is not materialised (scene_out->texels_rgba is
 * null), where every face's texels come from in the atlas (faces_out: 6 int32 per face — first texel in the pool, atlas
 * x, y, w, h, mirrored — for up to 72 faces), and per box whether no texel has alpha 0 (box_opaque_out[12]).  Only the
 * alpha bytes of the atlas are read.  What render_skin_batch does per skin before the device cuts the pool. */
int32_t mcskin_skin_layout(const uint8_t* atlas_rgba8, int32_t atlas_w, int32_t atlas_h, const float* pose12, McBox* boxes_out,
                           int32_t* faces_out, int32_t* n_faces_out, uint8_t* box_opaque_out, McScene* scene_out);
/* Batches of skins straight from their atlases (SkinParser::parse -> MeshBuilder::buildScene -> TileRenderer::render
 * per skin; skin_parser.cpp:11-132, mesh_builder.cpp:145-202): n_skins RGBA8 atlases of atlas_w x atlas_h (64x64 or
 * 64x32), one after the other in host memory, skin i -> image i of the device buffer(s).  poses12: 12 floats per skin
 * (rotX, rotZ in degrees for head, body, right arm, left arm, right leg, left leg) at a stride of pose_stride floats
 * (0: the same pose for every skin), or null for the standing pose.  The atlas is sliced into the scene's texel
 * pool on the DEVICE (16 KB per skin cross PCIe instead of 52 KB of float texels); the host only lays out the boxes,
 * from the alpha bytes.  Results equal mcskin_build_skin_scene + mcskin_cuda_context_render_batch bit for bit.
 * Asynchronous like render_batch. */
int32_t mcskin_cuda_context_render_skin_batch(McContext* ctx, const uint8_t* atlases_rgba8, int32_t atlas_w, int32_t atlas_h,
                                              int32_t n_skins, const float* poses12, int32_t pose_stride, const McConfig* cfg,
                                              void* d_out_f32, void* d_out_u8, void* stream);
/* The same, host to host and sharded by skin over devices 0..n_devices-1 of this process (BASELINE config 4):
 * skin i is rendered by device i % n_devices — scenes are independent frames, there is no exchange — one host
 * thread per device, image i lands at out_*[i] (n_scenes consecutive host images; either may be null).  Blocking. */
int32_t mcskin_cuda_render_batch_multi(const McScene* scenes, int32_t n_scenes, const McConfig* cfg, int32_t n_devices,
                                       float* out_rgba_f32, uint8_t* out_rgba_u8);

/* ---- PNG files made on the device ----
 * Every file is a valid PNG of one width x height 8-bit RGBA image (colour type 6, no interlace) holding only the
 * chunks IHDR, IDAT (one or more) and IEND, each with its CRC-32.  Its bytes are fixed by the image alone:
 *  - Row filters: each row takes the filter type (0 None .. 4 Paeth) whose filtered bytes, read as signed 8-bit
 *    values, have the smallest sum of absolute values (libpng's heuristic); on a tie the lower type.
 *  - Deflate: the filtered stream (per row its filter-type byte, then 4*width bytes) is cut into segments of
 *    32768 bytes, the last one shorter, each compressed on its own: no match reaches before its segment's start.  A
 *    segment is one block with dynamic Huffman codes of at most 15 bits (greedy LZ77 over a hash chain), or, when
 *    that would take more bytes than the segment has, one stored block.  Every segment then ends byte-aligned with
 *    an empty stored block (00 00 ff ff, pigz's sync-flush marker); the last segment's is the final block (BFINAL).
 *  - Segment k is the data of IDAT chunk k; the zlib header (78 01) opens the first, the Adler-32 of the filtered
 *    stream closes the last.
 * The same image gives the same bytes on every run, alone or at any place in a batch of any size. */

/* The largest file of a width x height image: every segment stored.  Host code, no device needed.  0 when width
 * or height is outside 1..65535. */
uint64_t mcskin_png_bound(int32_t width, int32_t height);
/* PNG files of n_images consecutive width x height RGBA8 images in device memory (the u8 layout render_batch and
 * render_skin_batch write), back to back into d_png (device, capacity bytes).  d_offsets (device, n_images + 1
 * uint64) receives the exclusive prefix sums of the file sizes: file i is bytes [d_offsets[i], d_offsets[i+1]) and
 * d_offsets[n_images] bytes in all, so one copy moves every file.  Asynchronous and ordered on `stream` (null: the
 * context's); the scratch is the context's and grows with the images encoded together (up to about 1 GiB, at least
 * one image).  MC_ERR_INVALID for a null pointer, a bad size or capacity < n_images * mcskin_png_bound. */
int32_t mcskin_cuda_context_encode_png(McContext* ctx, const void* d_rgba8, int32_t width, int32_t height, int32_t n_images,
                                       void* d_png, uint64_t capacity, uint64_t* d_offsets, void* stream);

/* ---- single-ray entry points: the reference's free functions, exercised through
 *      the same device code (no CPU fallback).  All arrays are HOST memory. ---- */
typedef struct McRay {
    float origin[3];
    float dir[3];
} McRay;

/* HitResult (src/scene/triangle.h:19-26) + the (box, face) id the reference does
 * not expose; tri_id = box*12 + face*2, -1 on miss. */
typedef struct McHit {
    int32_t hit;
    float t;
    float point[3];
    float normal[3];
    float tex_color[4];
    int32_t is_outer_layer;
    int32_t box;
    int32_t face;
} McHit;

/* intersectScene (intersection.cpp:408-421); box >= 0 restricts to intersectMesh of that box. */
int32_t mcskin_cuda_intersect(const McScene* scene, int32_t device, int32_t box,
                              const McRay* rays, int32_t n, McHit* out);
/* RayTracer::traceRay(ray, scene, depth, cfg->max_bounces, params, use_config ? &config : nullptr)
 * (raytracer.cpp:82-148). out_rgba: n*4 floats. */
int32_t mcskin_cuda_trace(const McScene* scene, const McConfig* cfg, int32_t device, int32_t use_config,
                          int32_t depth, const McRay* rays, int32_t n, float* out_rgba);
/* shade(hit, viewDir, light, scene, params, shadowFactor) (shading.cpp:62-96). */
int32_t mcskin_cuda_shade(const McScene* scene, const McConfig* cfg, int32_t device,
                          const McHit* hits, const float* view_dirs /* n*3 */, const float* shadow_factors /* n */,
                          int32_t n, float* out_rgba);
/* isInShadow(point, normal, lightPos, scene) (shading.cpp:14-26): out[i] = 0/1. */
int32_t mcskin_cuda_in_shadow(const McScene* scene, int32_t device, const float* points, const float* normals,
                              const float* light_positions, int32_t n, int32_t* out);
/* computeSoftShadow(point, normal, scene.light, scene, samples, seed) (shading.cpp:28-60). */
int32_t mcskin_cuda_soft_shadow(const McScene* scene, int32_t device, const float* points, const float* normals,
                                const uint32_t* seeds, int32_t samples, int32_t n, float* out);
/* RayTracer::computeAO(point, normal, scene, samples, radius, seed) (raytracer.cpp:38-78). */
int32_t mcskin_cuda_ambient_occlusion(const McScene* scene, int32_t device, const float* points,
                                      const float* normals, const uint32_t* seeds, int32_t samples,
                                      float radius, int32_t n, float* out);
/* Camera::generateRay(u, v, aspect) (camera.cpp:8-26). uv: n*2 floats. */
int32_t mcskin_cuda_generate_rays(const McScene* scene, int32_t device, float aspect, const float* uv,
                                  int32_t n, McRay* out);
/* RayTracer::backgroundColor(scene, u, v, use_config ? &config : nullptr) (raytracer.cpp:16-34). */
int32_t mcskin_cuda_background(const McScene* scene, const McConfig* cfg, int32_t device, int32_t use_config,
                               const float* uv, int32_t n, float* out_rgba);
/* std::sin / std::cos of float angles as the device evaluates them for the light-disk, lens and AO
 * samples (shading.cpp:51, tile_renderer.cpp:61-62, raytracer.cpp:62-64): bit-identical to glibc's
 * sinf / cosf on an FMA-capable x86-64 host for |angle| < 120. */
int32_t mcskin_cuda_sincos(int32_t device, const float* angles, int32_t n, float* out_sin, float* out_cos);
/* The same arithmetic evaluated on the host (no device needed): lets a CPU-only test pin the
 * restated algorithm to the host's libm. */
void mcskin_sincos_model(const float* angles, int32_t n, float* out_sin, float* out_cos);
/* std::pow(x, y) for floats as the device evaluates the Blinn-Phong exponent (shading.cpp:90):
 * bit-identical to glibc's powf on an FMA-capable x86-64 host for finite positive x and finite
 * non-zero y below the overflow threshold.  mcskin_powf_model is the same arithmetic on the host. */
int32_t mcskin_cuda_powf(int32_t device, const float* x, const float* y, int32_t n, float* out);
void mcskin_powf_model(const float* x, const float* y, int32_t n, float* out);
/* The launch order of the primary pass for the tile rows {first + k*stride} of a frame (no device needed):
 * block b renders part out_part[b] of out_parts[b] of local tile out_tile[b] (row-major in the band).  The
 * tiles that intersect the figure's screen rectangle come first and are split over parts_heavy blocks.
 * Returns the number of blocks, or a negative MC_ERR_*; fills at most `capacity` entries. */
int32_t mcskin_primary_launch_order(const McScene* scene, const McConfig* cfg, int32_t first_tile_row, int32_t stride,
                                    int32_t parts_heavy, int32_t parts_light, int32_t* out_tile, int32_t* out_part,
                                    int32_t* out_parts, int32_t capacity);
/* Measured ceiling of the roofline the bench reports against (SURVEY.md §8d): a kernel of independent,
 * unfused FADD / FMUL chains on every SM; returns the best of a few launches in lane-ops per second. */
int32_t mcskin_cuda_fp32_issue_peak(int32_t device, double* out_lane_ops_per_second);
/* Hit mask + triangle id of the pinhole ray through each pixel centre
 * (u=(px+.5)/W, v=(py+.5)/H): out_tri_id[py*W+px] = box*12+face*2, or -1. */
int32_t mcskin_cuda_aov(const McScene* scene, const McConfig* cfg, int32_t device, int32_t* out_tri_id);

/* ---- callers either side of the path (SURVEY §8f): skin atlas -> scene ---- */
/* Builds the flat scene the reference's SkinParser::parse + MeshBuilder::buildScene
 * produce for an RGBA8 atlas (64x64 or 64x32) and a pose (12 floats: rotX,rotZ for
 * head, body, rightArm, leftArm, rightLeg, leftLeg; NULL = standing).
 * (skin_parser.cpp:11-132, mesh_builder.cpp:66-202.)  Host-side, no GPU needed.
 * boxes_out: capacity 12; texels_out: capacity MCSKIN_MAX_SKIN_TEXELS*4 floats. */
#define MCSKIN_MAX_SKIN_BOXES 12
#define MCSKIN_MAX_SKIN_TEXELS 4096
int32_t mcskin_build_skin_scene(const uint8_t* atlas_rgba8, int32_t atlas_w, int32_t atlas_h,
                                const float* pose12, McBox* boxes_out, float* texels_out,
                                McScene* scene_out);

#ifdef __cplusplus
}
#endif
#endif /* MCSKIN_CUDA_H */
