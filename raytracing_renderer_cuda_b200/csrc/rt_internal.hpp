// rt_internal.hpp — the opaque handles of include/rt_api.h, shared by the translation units that implement the C-ABI (rt_api.cu:
// contexts, render entries; rt_scene.cu: scenes; rt_multi.cu: the multi-GPU entries; rt_selftest.cu: the primitives' tests).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>
#include <vector>

#include "../../include/rt_api.h"
#include "rt_error.hpp"
#include "rt_jpeg.cuh"
#include "rt_kernels.cuh"

// ends an rt_status function on a failing CUDA call, with the call and its place in the message
#define CUDA_TRY(expr)                                                                              \
    do {                                                                                              \
        cudaError_t e__ = (expr);                                                                     \
        if (e__ != cudaSuccess) {                                                                     \
            rtd::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__));   \
            return e__ == cudaErrorMemoryAllocation ? RT_ERR_OOM : RT_ERR_CUDA;                       \
        }                                                                                             \
    } while (0)

struct rt_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    int sm_count = 0;             // multiProcessorCount of the device (launch sizing)
    cudaMemPool_t pool = nullptr; // scene allocations (stream-ordered, private to the context)
    unsigned long long* d_ray_counter = nullptr;
    // the timing marks of one render entry: ev[0]..ev[1] the render (with stats), ev[1]..ev[2] the finalisation,
    // ev[2]..ev[3] the copy to the host
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    float4* accum = nullptr; // scratch for rt_render / rt_render_accum; the *_n fields count allocated elements
    size_t accum_n = 0;
    float* out_rgb = nullptr;
    size_t out_rgb_n = 0;
    rtd::WavefrontState* wf = nullptr;
    rtd::JpegState* jpg = nullptr; // device JPEG writer (rt_jpeg.cu), created on first use
    uint8_t* rgb8 = nullptr;       // flipped, quantised frame: input of the JPEG writer
    size_t rgb8_n = 0;
    // cudaArray allocations cost milliseconds; arrays of destroyed scenes are kept for the next scene of the
    // same image size (a frame loop that re-uploads its scene every frame then allocates nothing)
    struct CachedArray {
        int32_t width, height;
        cudaArray_t arr;
    };
    std::vector<CachedArray> array_cache;
    std::mutex cache_mutex; // a scene may be destroyed on one host thread while another creates the next one (frame pipelines)
};

struct rt_scene {
    rt_context* ctx = nullptr;
    rtd::DScene d{};
    rt_scene_info info{};
    std::vector<void*> allocs;
    std::vector<rt_context::CachedArray> arrays;
    std::vector<cudaTextureObject_t> texobjs;
    // what rt_scene_update needs of the creation description: the device index of every list ordinal, and the material
    // and texture counts
    std::vector<uint32_t> where;
    uint32_t n_materials = 0;
    uint32_t n_textures = 0;
    rtd::BvhNode4Q* nodes4q_mem = nullptr; // the quantised nodes' allocation, also when d.nodes4q is nullptr
    int* parents = nullptr; // parent of every inner node, then of every primitive (built on the first refit)
    uint32_t* where_dev = nullptr; // `where` on the device (built on the first rt_scene_update_device, from sph_c.w)
};

namespace rtd {
// the context's device and memory pool for the calling thread
inline rt_status make_current(const rt_context* ctx) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    set_thread_mempool(ctx->pool);
    return RT_OK;
}

// camera ctor (camera.h:7-31) in host float arithmetic
void make_camera(const rt_camera& c, DCamera& out);
} // namespace rtd

