// kernels.cuh — launch-side declarations shared by kernels.cu and the C-ABI host code.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <mutex>

#include "dev_types.cuh"
#include "host_prep.hpp"
#include "mcskin_cuda.h"

namespace mcskin {

constexpr int kBlockThreads = 256;
// scene blob staged per CTA (SceneBlobLayout: 212 boxes at most); with a kernel's own static shared memory it can pass
// the default 48 KB, so every kernel that stages it opts in to more (SmemOptIn)
constexpr unsigned int kMaxSceneSmemBytes = 40u * 1024u;

// Dynamic shared memory above the default 48 KB is an opt-in that CUDA keeps per function AND per
// device: a process that renders on several GPUs (mcskin_cuda_render_multi, one context per device)
// has to raise it on each of them.  One instance per group of kernels; limit() raises the attribute
// of every kernel of the group to the device's opt-in maximum (227 KB on sm_100) the first time it is
// called with that device current, and returns the bytes a launch may ask for (0: could not be raised,
// keep to kernels that fit 48 KB).
class SmemOptIn {
public:
    size_t limit(const void* const* fns, int nFns) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 0;
        std::lock_guard<std::mutex> lock(mu_);
        if (known_[dev]) return limit_[dev];
        int optin = 0;
        if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) optin = 0;
        bool ok = optin > 48 * 1024;
        // static + dynamic shared memory of a kernel may not exceed the opt-in maximum: the attribute is
        // the dynamic part, so each kernel's static bytes come off (asking for the full maximum is refused
        // with cudaErrorInvalidValue as soon as a kernel has one static __shared__ variable)
        int room = optin;
        for (int i = 0; ok && i < nFns; ++i) {
            cudaFuncAttributes fa{};
            ok = cudaFuncGetAttributes(&fa, fns[i]) == cudaSuccess;
            if (!ok) break;
            const int dyn = optin - static_cast<int>(fa.sharedSizeBytes);
            ok = dyn > 0 && cudaFuncSetAttribute(fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, dyn) == cudaSuccess;
            if (dyn < room) room = dyn;
        }
        if (!ok) cudaGetLastError();
        limit_[dev] = ok ? static_cast<size_t>(room) : 0;
        known_[dev] = true;
        return limit_[dev];
    }

private:
    static constexpr int kMaxDevices = 64;
    std::mutex mu_;
    size_t limit_[kMaxDevices] = {};
    bool known_[kMaxDevices] = {};
};

// Which tiles of the frame a launch covers, and where its pixels land.
// Row form (tile_map == null): local tile row r is frame tile row first_tile_row + r*tile_row_stride and lands
// at tile row out_first_row + r*out_row_stride of the output image (0 and 1 for a compact band of those rows;
// a frame split over several streams writes interleaved rows of one shared band image; out = frame row for a
// full-frame image).
// Map form (tile_map != null): local tile t is frame tile tile_map[t] (= ty*tiles_x + tx), any set of whole
// tiles, the ones that intersect the figure's screen rectangle first (n_heavy of them); the output image is a
// full frame and every tile lands at its own place.
struct BandView {
    int first_tile_row, tile_row_stride, n_tile_rows;
    int out_first_row, out_row_stride;
    float4* out_f32;  // may be null
    uchar4* out_u8;   // may be null
    // If set: the image the tiles that intersect the figure's screen rectangle are written to instead (same
    // layout).  The host API points these at the caller's page-locked image (mapped into the device address space),
    // so that the pixels that are final only when the frame ends need no copy afterwards, while the background
    // tiles — final after the primary pass — go to device memory and leave by DMA next to the shading kernels.
    float4* hot_f32;
    uchar4* hot_u8;
    const int* tile_map;  // device memory, or null
    int n_tiles, n_heavy;
    // != 0: the shaded pixels land in memory across PCIe or NVLink (a mapped host image, a peer GPU's frame): the
    // resolve kernel then stores runs of neighbouring pixels together instead of one pixel at a time
    int far_output;
    // diagnosis ("debug_primary_timing" option): 4 words per block of the pixel-per-lane primary kernels —
    // %globaltimer at entry and exit, the block's frame tile, part | parts << 16; null otherwise
    unsigned long long* block_times;
};
// tiles of a band
__host__ __device__ inline int band_tile_count(const BandView& band, int tilesX) {
    return band.tile_map ? band.n_tiles : band.n_tile_rows * tilesX;
}
// AOV planes (McAovTargets, device pointers) travel next to a BandView, indexed like its out_f32: the launchers pick the
// AOV instantiations of the shading kernels when any plane is set, and the kernels of frames without run as before.
// (Not members of BandView: the batched primary kernels copy a scene's BandView, and a larger one costs them registers.)
__host__ __device__ inline bool aov_any(const McAovTargets* a) {
    return a && (a->coverage || a->depth || a->tri_id || a->normal || a->albedo);
}
// the guide planes (normal, albedo): they need the camera ray's normal and texel colour as well as its distance and id
__host__ __device__ inline bool aov_guides(const McAovTargets& a) { return a.normal || a.albedo; }

// Work list produced by the primary pass for the shading pass.
struct ActiveList {
    unsigned int* count;  // number of slots in use (device counter)
    uint2* slot_pixel;    // x = index into the band image, y = px | (py << 16); x = 0xffffffff: unused slot
    float* records;       // slot-major, spp * draws_per_sample floats per slot: jx, jy [, lens r1, r2]
    unsigned int capacity;
    unsigned int* count_host;  // if set (page-locked host memory as the device sees it): the frame's last kernel leaves the count there
};

struct FramePointers {
    const unsigned char* blob;  // SceneBlobLayout image (device memory)
    const float4* texels;
    unsigned int blob_bytes;
};

// ---- launchers that exist in both builds of the kernels (mcskin:: for any scene, mcskin::plain:: for scenes
//      without posed boxes; dev_types.cuh) ----
#define MCSKIN_HOT_KERNEL_LAUNCHERS                                                                                      \
    bool launch_primary(const DevFrame& fr, const FramePointers& fp, const BandView& band, const ActiveList& list,      \
                        int classify, uint32_t* tileStates, bool seedTiles, int primaryTargetBlocks, int heavyTargetTiles, \
                        cudaStream_t stream);                                                                           \
    int launch_shade(const DevFrame& fr, const FramePointers& fp, const BandView& band, const ActiveList& list,         \
                     int gridBlocks, unsigned int* groupCounter, unsigned int firstSlot, cudaStream_t stream,           \
                     int variant = 1, const McAovTargets* aov = nullptr);
// Primary pass: per-tile jitter stream, camera rays, hit/miss classification, background
// resolve of pixels no sample of which hits, work records for the rest.
// classify == 0 puts every pixel on the work list (used for spp > 256 and for tests).
// tileStates: scratch of 624 words per tile of the band (seeded engine states).
// seedTiles: false when tileStates already holds the states of exactly these tiles (they depend on
// the image width, the tile size and the tile rows of the band only, not on the scene).
// primaryTargetBlocks: tiles are split over several blocks until the launch has about this many.
// Returns true when tileStates holds the seeded engines of the band's tiles afterwards.
// heavyTargetTiles: the tiles that intersect the figure are split over more blocks while the launch has
// fewer tiles than this.
MCSKIN_HOT_KERNEL_LAUNCHERS
namespace plain {
MCSKIN_HOT_KERNEL_LAUNCHERS
}
namespace counter {
MCSKIN_HOT_KERNEL_LAUNCHERS
}
// Shading pass: full integrator for every sample of every listed pixel, ordered resolve.
// aov: the AOV planes of the listed pixels too (a second, small kernel).  Returns the kernels launched.
// Megakernel form of the shading pass over the listed pixels from `firstSlot` on.
// variant 1: block-synchronous groups; variant 2: warp-autonomous groups with dynamic
// distribution (groupCounter: a zeroed device counter; spp must be a power of two <= 32).

// Engine states the pixel-per-lane primary kernels keep per tile for a launch of nTiles tiles x nScenes scenes: 1 (the
// seed) when no tile is split over blocks, else one per round of 256 pixels.  tileStates must hold nTiles * this * 624
// words.  (Host arithmetic, the same for every build of the kernels.)
inline int primary_states_per_tile(const DevFrame& fr, int nTiles, int nScenes, int primaryTargetBlocks, int heavyTargetTiles) {
    if (nTiles <= 0 || fr.draws_per_sample <= 0) return 1;
    const int roundsPerTile = (fr.tile_size * fr.tile_size + kBlockThreads - 1) / kBlockThreads;
    const long long allTiles = static_cast<long long>(nTiles) * std::max(1, nScenes);
    const bool split = primaryTargetBlocks > allTiles || heavyTargetTiles > allTiles;
    return split && roundsPerTile > 1 ? roundsPerTile : 1;
}

// Single-query views of the same device code (all pointers are device memory).
void launch_intersect(const DevFrame& fr, const FramePointers& fp, int box, const McRay* rays, int n, McHit* out,
                      cudaStream_t stream);
void launch_trace(const DevFrame& fr, const FramePointers& fp, int depth, const McRay* rays, int n, float4* out,
                  cudaStream_t stream);
void launch_shade_hits(const DevFrame& fr, const FramePointers& fp, const McHit* hits, const float* viewDirs,
                       const float* shadowFactors, int n, float4* out, cudaStream_t stream);
void launch_in_shadow(const DevFrame& fr, const FramePointers& fp, const float* points, const float* normals,
                      const float* lights, int n, int* out, cudaStream_t stream);
void launch_soft_shadow(const DevFrame& fr, const FramePointers& fp, const float* points, const float* normals,
                        const uint32_t* seeds, int samples, int n, float* out, cudaStream_t stream);
void launch_ambient_occlusion(const DevFrame& fr, const FramePointers& fp, const float* points, const float* normals,
                              const uint32_t* seeds, int samples, float radius, int n, float* out,
                              cudaStream_t stream);
void launch_generate_rays(const DevFrame& fr, const float* uv, int n, McRay* out, cudaStream_t stream);
void launch_background(const DevFrame& fr, const float* uv, int n, float4* out, cudaStream_t stream);
// Host evaluation of the primary pass's block -> (tile, part) map for a band (the same functions the
// kernels run): returns the number of blocks, fills at most `capacity` entries.
int primary_launch_order(const DevFrame& fr, int first, int stride, int partsHeavy, int partsLight, int* outTile,
                         int* outPart, int* outParts, int capacity);
// FADD/FMUL issue-rate microbenchmark: `iters` rounds of 16 unfused operations per thread; result written to sink
void launch_fp32_peak(int blocks, int iters, float* sink, cudaStream_t stream);
void launch_peer_signal(unsigned int* flag, unsigned int value, cudaStream_t stream);
void launch_peer_wait(const unsigned int* flags, int n, unsigned int value, unsigned int* timedOut, cudaStream_t stream);
void launch_powf(const float* x, const float* y, int n, float* out, cudaStream_t stream);
void launch_sincos(const float* angles, int n, float* outSin, float* outCos, cudaStream_t stream);
void launch_aov(const DevFrame& fr, const FramePointers& fp, int* outTriId, cudaStream_t stream);

// Skin slicing on the device (SkinParser::parse, skin_parser.cpp:11-110): one job per skin.
struct SkinSliceJob {
    const uchar4* atlas;            // raw RGBA8 atlas, atlasW x atlasH
    const SkinFaceSource* faces;    // where every face's texels come from (host_prep.hpp)
    float4* texels;                 // the scene's pool: nTexels texels, then the two synthetic ones
    int atlasW, atlasH, nFaces, nTexels;
};
// records: nSkins staging records of recordStride bytes in device memory, each with its SkinSliceJob at jobOffset
void launch_slice_skins(const unsigned char* records, size_t recordStride, size_t jobOffset, int nSkins, cudaStream_t stream);

}  // namespace mcskin
