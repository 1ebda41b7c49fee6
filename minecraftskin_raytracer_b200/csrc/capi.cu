// capi.cu — the extern "C" layer of include/mcskin_cuda.h: the single-query entry points, host memory, IPC and peer
// utilities.  The units next to it hold the rest (capi_internal.hpp).  No exceptions leave this layer; every failure is a
// negative MC_ERR_* plus a thread-local message (mcskin_cuda_last_error).
#include <cstring>
#include "capi_internal.hpp"

namespace {

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
    return upload_scene(*ctx);
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
