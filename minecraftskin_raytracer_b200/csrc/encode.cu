// encode.cu — PNG files of device images (the C ABI over png.cu): argument checks, the context's scratch, groups.
#include "capi_internal.hpp"
#include "png.cuh"

namespace {

// scratch kept per launch group: a group's filtered streams, tokens and segments stay within this many bytes
// (a group always holds at least one image)
constexpr uint64_t kScratchBudget = 1ull << 30;

uint64_t align256(uint64_t v) { return (v + 255) & ~255ull; }

}  // namespace

extern "C" {

uint64_t mcskin_png_bound(int32_t width, int32_t height) { return png::file_bound(width, height); }

int32_t mcskin_cuda_context_encode_png(McContext* ctx, const void* d_rgba8, int32_t width, int32_t height, int32_t n_images,
                                       void* d_png, uint64_t capacity, uint64_t* d_offsets, void* stream) {
    if (!ctx || n_images < 0 || !d_offsets) return fail(MC_ERR_INVALID, "encode_png: bad argument");
    const uint64_t bound = png::file_bound(width, height);
    if (bound == 0)
        return fail(MC_ERR_INVALID, "encode_png: bad image size " + std::to_string(width) + "x" + std::to_string(height));
    if (n_images > 0 && (!d_rgba8 || !d_png)) return fail(MC_ERR_INVALID, "encode_png: null image or output");
    if (capacity / bound < static_cast<uint64_t>(n_images))
        return fail(MC_ERR_INVALID, "encode_png: capacity " + std::to_string(capacity) + " is under n_images * mcskin_png_bound = " +
                                        std::to_string(n_images) + " * " + std::to_string(bound));
    CU_TRY(cudaSetDevice(ctx->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
    if (n_images == 0) {
        CU_TRY(cudaMemsetAsync(d_offsets, 0, sizeof(uint64_t), s));
        return MC_OK;
    }
    const uint64_t stride = png::filtered_stride(width, height), nSeg = png::segments(width, height);
    const uint64_t perImage = align256(stride) + align256(nSeg * png::kSegBytes * sizeof(uint32_t)) + align256(nSeg * png::kSlotBytes) +
                              align256(nSeg * sizeof(uint32_t)) + align256(nSeg * sizeof(uint2)) +
                              align256(nSeg * sizeof(unsigned long long)) + 256;
    const uint64_t maxGroup = std::min<uint64_t>(static_cast<uint64_t>(n_images), 0x7fffffffull / nSeg);
    if (maxGroup == 0) return fail(MC_ERR_INVALID, "encode_png: image has too many segments");
    const int group = static_cast<int>(std::max<uint64_t>(1, std::min<uint64_t>(maxGroup, kScratchBudget / perImage)));
    const uint64_t g = static_cast<uint64_t>(group);
    // one allocation carved into the group's arrays (each 256-byte aligned)
    const uint64_t sizes[7] = {align256(g * stride), align256(g * nSeg * png::kSegBytes * sizeof(uint32_t)), align256(g * nSeg * png::kSlotBytes),
                               align256(g * nSeg * sizeof(uint32_t)), align256(g * nSeg * sizeof(uint2)),
                               align256(g * nSeg * sizeof(unsigned long long)), align256(g * sizeof(uint32_t))};
    uint64_t total = 0;
    for (uint64_t v : sizes) total += v;
    CU_TRY(ctx->pngScratch.reserve(total));
    unsigned char* at = static_cast<unsigned char*>(ctx->pngScratch.p);
    unsigned char* parts[7];
    for (int i = 0; i < 7; ++i) {
        parts[i] = at;
        at += sizes[i];
    }
    const png::Scratch scratch{parts[0], reinterpret_cast<uint32_t*>(parts[1]), parts[2], reinterpret_cast<uint32_t*>(parts[3]),
                               reinterpret_cast<uint2*>(parts[4]), reinterpret_cast<unsigned long long*>(parts[5]),
                               reinterpret_cast<uint32_t*>(parts[6])};
    const size_t imageBytes = static_cast<size_t>(width) * height * 4;
    for (int i0 = 0; i0 < n_images; i0 += group) {
        const int n = std::min(group, n_images - i0);
        const cudaError_t e = png::encode(static_cast<const uint8_t*>(d_rgba8) + i0 * imageBytes, width, height, n, scratch,
                                          static_cast<uint8_t*>(d_png), reinterpret_cast<unsigned long long*>(d_offsets) + i0, i0 == 0, s);
        if (e != cudaSuccess) return cuda_fail(e, "encode_png");
    }
    return MC_OK;
}

}  // extern "C"
