// rt_selftest.cu — self-test entries of the device primitives of rt_prims.cuh (include/rt_api.h): host arrays in, host
// arrays out, so a test can compare prims::exclusive_sum and prims::sort_pairs_u64_u32 with a host reference at any size.
// Every device buffer the primitives may write sits between two guard regions, and the buffers are allocated with the
// sizing helpers the library's own callers use (scan_scratch_elems, sort_scratch_elems): a write past a buffer, or a
// scratch size that is too small, shows up as a changed guard byte.  The whole allocation, payload included, starts as
// 0xA5 bytes, so a read of scratch the primitive never wrote gives the same wrong answer on every run.
// The primitives are templates and static kernels, so this translation unit gets its own copies and leaves the code of
// the other units unchanged.
#include <cstdarg>
#include <cstdio>
#include <exception>
#include <new>
#include <vector>

#include "rt_internal.hpp"
#include "rt_prims.cuh"

namespace {

constexpr size_t kGuard = 256;     // bytes before and after every buffer
constexpr unsigned char kFill = 0xA5;

void fail(const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    rtd::set_error_message(buf);
}
#define S_ARG(cond, msg)                       \
    do {                                       \
        if (!(cond)) {                         \
            fail("invalid argument: %s", msg); \
            return RT_ERR_INVALID_ARG;         \
        }                                      \
    } while (0)
#define S_CATCH                                     \
    catch (const std::bad_alloc&) {                 \
        fail("out of host memory");                 \
        return RT_ERR_OOM;                          \
    }                                               \
    catch (const std::exception& e) {               \
        fail("unexpected exception: %s", e.what()); \
        return RT_ERR_INVALID_ARG;                  \
    }

// The device buffers of one call, from the context's pool, each between two kGuard-byte guards; freed on the stream when
// the call returns.  The first error sticks in `e` and turns every later step into a no-op.
struct Guarded {
    cudaStream_t st;
    cudaError_t e = cudaSuccess;
    std::vector<std::pair<unsigned char*, size_t>> bufs; // allocation, payload bytes

    explicit Guarded(cudaStream_t s) : st(s) {}
    ~Guarded() {
        for (auto& b : bufs) cudaFreeAsync(b.first, st);
    }
    template <class T>
    T* alloc(size_t count) {
        unsigned char* p = nullptr;
        const size_t bytes = count * sizeof(T);
        if (e == cudaSuccess) e = rtd::malloc_async(&p, bytes + 2 * kGuard, st);
        if (e != cudaSuccess) return nullptr;
        bufs.push_back({p, bytes});
        e = cudaMemsetAsync(p, kFill, bytes + 2 * kGuard, st);
        return reinterpret_cast<T*>(p + kGuard); // (kGuard keeps the allocation's alignment)
    }
    void copy(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
        if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(dst, src, bytes, kind, st);
    }
    // synchronises; *overrun = 1 when any guard byte of any buffer changed
    void check_guards(int32_t* overrun) {
        std::vector<unsigned char> h(2 * kGuard * bufs.size());
        for (size_t k = 0; k < bufs.size(); ++k) {
            copy(&h[2 * k * kGuard], bufs[k].first, kGuard, cudaMemcpyDeviceToHost);
            copy(&h[(2 * k + 1) * kGuard], bufs[k].first + kGuard + bufs[k].second, kGuard, cudaMemcpyDeviceToHost);
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        int32_t bad = 0;
        for (unsigned char c : h) bad |= c != kFill;
        *overrun = bad;
    }
};

rt_status finish(const Guarded& g, const char* entry) {
    if (g.e == cudaSuccess) return RT_OK;
    fail("%s: %s", entry, cudaGetErrorString(g.e));
    return g.e == cudaErrorMemoryAllocation ? RT_ERR_OOM : RT_ERR_CUDA;
}

rt_status make_current(const rt_context* ctx) {
    const cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) {
        fail("cudaSetDevice(%d): %s", ctx->device, cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    rtd::set_thread_mempool(ctx->pool);
    return RT_OK;
}

template <class T>
rt_status scan(rt_context* ctx, const void* in, void* out, size_t n, bool in_place, int32_t* overrun) {
    Guarded g(ctx->stream);
    T* d_out = g.alloc<T>(n);
    T* d_in = in_place ? d_out : g.alloc<T>(n);
    T* scratch = g.alloc<T>(rtd::prims::scan_scratch_elems(n));
    g.copy(d_in, in, n * sizeof(T), cudaMemcpyHostToDevice);
    if (g.e == cudaSuccess) g.e = rtd::prims::exclusive_sum<T>(d_in, d_out, n, scratch, g.st);
    g.copy(out, d_out, n * sizeof(T), cudaMemcpyDeviceToHost);
    g.check_guards(overrun);
    return finish(g, "rt_selftest_exclusive_sum");
}

} // namespace

extern "C" rt_status rt_selftest_exclusive_sum(rt_context* ctx, const void* in, void* out, size_t n, int32_t elem_bytes,
                                               int32_t in_place, int32_t* overrun) try {
    S_ARG(ctx && overrun, "ctx/overrun is NULL");
    S_ARG(n == 0 || (in && out), "in/out is NULL");
    S_ARG(elem_bytes == 4 || elem_bytes == 8, "elem_bytes must be 4 or 8");
    *overrun = 0;
    if (n == 0) return RT_OK;
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    return elem_bytes == 4 ? scan<uint32_t>(ctx, in, out, n, in_place != 0, overrun)
                           : scan<unsigned long long>(ctx, in, out, n, in_place != 0, overrun);
} S_CATCH

extern "C" rt_status rt_selftest_sort_pairs(rt_context* ctx, const uint64_t* keys, const uint32_t* vals, size_t n, int32_t passes,
                                            uint64_t* keys_out, uint32_t* vals_out, int32_t* in_alt, int32_t* overrun) try {
    S_ARG(ctx && in_alt && overrun, "ctx/in_alt/overrun is NULL");
    S_ARG(n == 0 || (keys && vals && keys_out && vals_out), "keys/vals/keys_out/vals_out is NULL");
    S_ARG(passes >= 1 && passes <= 8, "passes must be in [1, 8]");
    S_ARG(n <= UINT32_MAX, "n must fit in 32 bits");
    *in_alt = 0;
    *overrun = 0;
    if (n == 0) return RT_OK;
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    Guarded g(ctx->stream);
    unsigned long long* k = g.alloc<unsigned long long>(n);
    uint32_t* v = g.alloc<uint32_t>(n);
    unsigned long long* k_alt = g.alloc<unsigned long long>(n);
    uint32_t* v_alt = g.alloc<uint32_t>(n);
    uint32_t* scratch = g.alloc<uint32_t>(rtd::prims::sort_scratch_elems(n));
    g.copy(k, keys, n * sizeof(uint64_t), cudaMemcpyHostToDevice);
    g.copy(v, vals, n * sizeof(uint32_t), cudaMemcpyHostToDevice);
    bool alt = false;
    if (g.e == cudaSuccess) g.e = rtd::prims::sort_pairs_u64_u32(k, v, k_alt, v_alt, uint32_t(n), passes, scratch, &alt, g.st);
    g.copy(keys_out, alt ? k_alt : k, n * sizeof(uint64_t), cudaMemcpyDeviceToHost);
    g.copy(vals_out, alt ? v_alt : v, n * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    g.check_guards(overrun);
    *in_alt = alt ? 1 : 0;
    return finish(g, "rt_selftest_sort_pairs");
} S_CATCH
