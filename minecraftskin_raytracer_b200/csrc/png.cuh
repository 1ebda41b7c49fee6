// png.cuh — PNG files on the device (png.cu): row filters, segmented deflate, chunk layout and checksums.
#pragma once
#include <cstddef>
#include <cstdint>

#include <cuda_runtime.h>

namespace mcskin {
namespace png {

// The filtered stream of an image (one filter-type byte + 4*width bytes per row) is cut into segments of this many
// bytes, each deflated on its own: a single stored block holds one (LEN <= 65535), and no distance can exceed the
// 32 KiB window.
constexpr uint32_t kSegBytes = 32768;
// Bytes one segment may take in its slot: the stored form, a 5-byte block header plus the 5-byte empty stored block.
constexpr uint32_t kSlotBytes = kSegBytes + 16;
constexpr int32_t kMaxSide = 65535;

// Filtered bytes of one image, and that length rounded up to 16 (the stride of images in the filtered buffer).
inline uint64_t filtered_bytes(int32_t w, int32_t h) { return static_cast<uint64_t>(h) * (4ull * static_cast<uint64_t>(w) + 1); }
inline uint64_t filtered_stride(int32_t w, int32_t h) { return (filtered_bytes(w, h) + 15) & ~15ull; }
inline uint64_t segments(int32_t w, int32_t h) { return (filtered_bytes(w, h) + kSegBytes - 1) / kSegBytes; }
// Size of the file when every segment is stored: signature 8, IHDR 25, per segment an IDAT chunk (12) holding a
// stored block (5) and the empty stored block (5), zlib header 2 and Adler-32 4, IEND 12.  0 for a bad size.
inline uint64_t file_bound(int32_t w, int32_t h) {
    if (w < 1 || h < 1 || w > kMaxSide || h > kMaxSide) return 0;
    return 8 + 25 + 2 + 4 + 12 + filtered_bytes(w, h) + 22 * segments(w, h);
}

// The scratch of one launch group of n images (device pointers; sizes from the functions above).
struct Scratch {
    uint8_t* filtered;        // n * filtered_stride
    uint32_t* tokens;         // n * segments * kSegBytes: the LZ77 tokens of every segment
    uint8_t* slots;           // n * segments * kSlotBytes: every segment's deflate bytes
    uint32_t* segBytes;       // n * segments
    uint2* segAdler;          // n * segments: (sum of bytes, sum of bytes weighted by distance to the end) mod 65521
    unsigned long long* segOff;  // n * segments: where the segment's IDAT chunk starts in its file
    uint32_t* imgAdler;       // n
};

// The four launches that turn n consecutive RGBA8 images into n PNG files back to back at png + offsets[0],
// offsets[1..n] = offsets[0] + the running file sizes.  offsets[0] must hold the start when `first` is false (it is
// the previous group's end); `first` writes 0 there.
cudaError_t encode(const uint8_t* rgba, int32_t w, int32_t h, int32_t n, const Scratch& s, uint8_t* png,
                   unsigned long long* offsets, bool first, cudaStream_t stream);

}  // namespace png
}  // namespace mcskin
