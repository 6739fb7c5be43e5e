// host_util.h — host-side plumbing shared by the engine's units: the thread-local error string behind mb_last_error,
// the MB_CUDA / MB_TRY status macros, device buffers, pointer classification, per-category event timing and the
// runtime-value -> template-constant dispatch used at every templated launch site.
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/mollyb200.h"

namespace mb {

static thread_local std::string g_last_error;
static int set_error(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

#define MB_CUDA(call)                                                                                  \
    do {                                                                                               \
        cudaError_t err__ = (call);                                                                    \
        if (err__ != cudaSuccess) {                                                                    \
            return set_error(MB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(err__) + " (" + \
                                              __FILE__ + ":" + std::to_string(__LINE__) + ")");        \
        }                                                                                              \
    } while (0)
#define MB_TRY(expr)                 \
    do {                             \
        int rc__ = (expr);           \
        if (rc__ != MB_OK) return rc__; \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    ~DevBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
    cudaError_t ensure(size_t nbytes) {
        if (nbytes <= bytes) return cudaSuccess;
        release();
        cudaError_t e = cudaMalloc(&p, nbytes);
        if (e == cudaSuccess) bytes = nbytes;
        return e;
    }
    template <typename U>
    U* as() const {
        return reinterpret_cast<U*>(p);
    }
};

static bool is_device_ptr(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Runtime value -> compile-time constant. dispatch(flag, f) calls f(std::true_type / std::false_type);
// dispatch(Vals<V...>{}, v, f) calls f(std::integral_constant<int, V>) for the V equal to v. Only the listed values are
// instantiated, so the lists decide which kernel variants exist; a value outside the list is an MB_ERR_INVALID.
template <int... Vs>
struct Vals {};
template <typename F>
int dispatch(bool flag, F&& f) {
    return flag ? f(std::true_type{}) : f(std::false_type{});
}
template <int... Vs, typename F>
int dispatch(Vals<Vs...>, int v, F&& f, const char* missing = "no kernel variant for this configuration") {
    int rc = MB_OK;
    const bool found = ((v == Vs && (rc = f(std::integral_constant<int, Vs>{}), true)) || ...);
    return found ? rc : set_error(MB_ERR_INVALID, missing);
}

// Optional per-category device timing with CUDA events on the engine's stream (mb_set_profiling).
struct Prof {
    enum { FORCE = 0, VV = 1, REBUILD = 2, NCAT = 3 };
    bool enabled = false;
    cudaStream_t stream = nullptr;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev[NCAT];
    size_t used[NCAT] = {0, 0, 0};
    double ms[NCAT] = {0, 0, 0};
    long long count[NCAT] = {0, 0, 0};
    ~Prof() {
        for (int c = 0; c < NCAT; c++)
            for (auto& p : ev[c]) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
    }
    void begin(int c) {
        if (!enabled) return;
        if (used[c] == ev[c].size()) {
            if (ev[c].size() >= 8192) { collect(); }
            if (used[c] == ev[c].size()) {
                cudaEvent_t a, b;
                cudaEventCreate(&a);
                cudaEventCreate(&b);
                ev[c].emplace_back(a, b);
            }
        }
        cudaEventRecord(ev[c][used[c]].first, stream);
    }
    void end(int c) {
        if (!enabled) return;
        cudaEventRecord(ev[c][used[c]].second, stream);
        used[c]++;
    }
    void collect() {
        cudaStreamSynchronize(stream);
        for (int c = 0; c < NCAT; c++) {
            for (size_t k = 0; k < used[c]; k++) {
                float t = 0;
                if (cudaEventElapsedTime(&t, ev[c][k].first, ev[c][k].second) == cudaSuccess) { ms[c] += t; count[c]++; }
            }
            used[c] = 0;
        }
    }
    void reset() {
        collect();
        for (int c = 0; c < NCAT; c++) { ms[c] = 0; count[c] = 0; }
    }
};

}  // namespace mb
