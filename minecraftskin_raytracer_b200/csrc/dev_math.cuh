// dev_math.cuh — the reference's Vec3/Color arithmetic with its exact rounding.
//
// The parity-critical chain (ray generation -> slab test -> hit point -> UV ->
// texel -> shadow seed -> reflection) must round exactly like the reference built
// for x86-64 without FMA: every product and sum is a separate IEEE operation, in the
// reference's order (src/math/vec3.h:6-51).  This translation unit is therefore
// compiled with --fmad=false and default IEEE division / sqrt (no -use_fast_math);
// fused operations appear only where they are written explicitly (fmaf) in colour
// math that never feeds back into geometry.
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

namespace mcskin {

struct V3 {
    float x, y, z;
};

__device__ __forceinline__ V3 mk3(float x, float y, float z) { return V3{x, y, z}; }
__device__ __forceinline__ V3 ld3(const float* p) { return V3{p[0], p[1], p[2]}; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 operator*(V3 a, float s) { return V3{a.x * s, a.y * s, a.z * s}; }
__device__ __forceinline__ float dot3(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 cross3(V3 a, V3 b) {
    return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
__device__ __forceinline__ float len3(V3 a) { return sqrtf(a.x * a.x + a.y * a.y + a.z * a.z); }
// vec3.h:22 — v / s multiplies by the rounded reciprocal
__device__ __forceinline__ V3 div3(V3 a, float s) {
    const float inv = 1.0f / s;
    return V3{a.x * inv, a.y * inv, a.z * inv};
}
// vec3.h:46-50
__device__ __forceinline__ V3 normalize3(V3 a) {
    const float l = len3(a);
    if (l < 1e-8f) return V3{0.0f, 0.0f, 0.0f};
    return div3(a, l);
}

// std::clamp(v, lo, hi)
__device__ __forceinline__ float clampf(float v, float lo, float hi) { return (v < lo) ? lo : (hi < v) ? hi : v; }
__device__ __forceinline__ float clamp01(float v) { return clampf(v, 0.0f, 1.0f); }

__device__ __forceinline__ float4 clamp4(float4 c) {
    return make_float4(clamp01(c.x), clamp01(c.y), clamp01(c.z), clamp01(c.w));
}

// x86-64 gcc lowers static_cast<unsigned>(float) to a 64-bit cvttss2si and keeps the
// low 32 bits: negatives wrap, |f| >= 2^63 and NaN give 0 (raytracer.cpp:110-112,
// SURVEY.md §7 "hard parts").  CUDA's own float->unsigned saturates, so go through
// int64 by hand.
__device__ __forceinline__ uint32_t seed_cast(float f) {
    if (!(f > -9.2233720368547758e18f && f < 9.2233720368547758e18f)) return 0u;
    return static_cast<uint32_t>(static_cast<unsigned long long>(__float2ll_rz(f)));
}

// A colour channel as the reference stores it.  With finite inputs every NaN the reference makes comes from its own
// arithmetic (0.0f / 0.0f in computeAO with no samples, ks * inf * 0 in shade() with a negative shininess), where x86
// gives the default NaN 0xffc00000 and each later operation passes it on unchanged; NVIDIA GPUs give 0x7fffffff.  So a
// NaN leaves the device as 0xffc00000.  NaN payloads carried in by the inputs (NaN texels or config values) are not
// reproduced.
__device__ __forceinline__ float x86_nan(float c) { return c == c ? c : __uint_as_float(0xffc00000u); }
__device__ __forceinline__ float4 x86_nan4(float4 c) {
    return make_float4(x86_nan(c.x), x86_nan(c.y), x86_nan(c.z), x86_nan(c.w));
}

// uint8(clamp(c)*255 + 0.5) (image_writer.cpp:18-22)
__device__ __forceinline__ uint32_t quantize8(float c) {
    return static_cast<uint32_t>(__float2int_rz(clamp01(c) * 255.0f + 0.5f)) & 0xffu;
}
__device__ __forceinline__ uchar4 quantize4(float4 c) {
    return make_uchar4(static_cast<unsigned char>(quantize8(c.x)), static_cast<unsigned char>(quantize8(c.y)),
                       static_cast<unsigned char>(quantize8(c.z)), static_cast<unsigned char>(quantize8(c.w)));
}

}  // namespace mcskin
