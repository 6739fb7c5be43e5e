// dynlib.h — NCCL and cuFFT, bound at run time (dlopen) so that single-GPU users do not need NCCL and only PME systems
// need cuFFT. Only the entry points the engine calls are declared.
#pragma once
#include <dlfcn.h>

#include "host_util.h"

namespace mb {

// NCCL: only what the decomposed step uses: point-to-point halo exchange, grouped broadcasts, one tiny all-reduce.
extern "C" {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef enum { ncclSuccess = 0 } ncclResult_t;
typedef enum { ncclInt8 = 0, ncclChar = 0, ncclFloat64 = 8, ncclDouble = 8 } ncclDataType_t;
typedef enum { ncclSum = 0 } ncclRedOp_t;
}

#define MB_SYM(field, name) field = reinterpret_cast<decltype(field)>(dlsym(lib, name)); if (!field) return false

struct Nccl {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool load() {
        if (lib) return true;
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return false;
        MB_SYM(GetUniqueId, "ncclGetUniqueId");
        MB_SYM(CommInitRank, "ncclCommInitRank");
        MB_SYM(CommDestroy, "ncclCommDestroy");
        MB_SYM(GroupStart, "ncclGroupStart");
        MB_SYM(GroupEnd, "ncclGroupEnd");
        MB_SYM(Send, "ncclSend");
        MB_SYM(Recv, "ncclRecv");
        MB_SYM(Broadcast, "ncclBroadcast");
        MB_SYM(AllReduce, "ncclAllReduce");
        MB_SYM(AllGather, "ncclAllGather");
        MB_SYM(GetErrorString, "ncclGetErrorString");
        return true;
    }
};
static Nccl g_nccl;

// cuFFT: plain library FFT; the spreading, convolution and interpolation kernels around it are ours (pme.cuh).
struct Cufft {
    void* lib = nullptr;
    int (*Plan3d)(int*, int, int, int, int) = nullptr;
    int (*SetStream)(int, cudaStream_t) = nullptr;
    int (*ExecC2C)(int, void*, void*, int) = nullptr;
    int (*ExecZ2Z)(int, void*, void*, int) = nullptr;
    int (*Destroy)(int) = nullptr;
    bool load() {
        if (lib) return true;
        lib = dlopen("libcufft.so.11", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libcufft.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return false;
        MB_SYM(Plan3d, "cufftPlan3d");
        MB_SYM(SetStream, "cufftSetStream");
        MB_SYM(ExecC2C, "cufftExecC2C");
        MB_SYM(ExecZ2Z, "cufftExecZ2Z");
        MB_SYM(Destroy, "cufftDestroy");
        return true;
    }
};
static Cufft g_cufft;
#undef MB_SYM

#define MB_NCCL(call)                                                                                       \
    do {                                                                                                    \
        ncclResult_t r__ = (call);                                                                          \
        if (r__ != ncclSuccess)                                                                             \
            return set_error(MB_ERR_CUDA, std::string(#call) + ": " + g_nccl.GetErrorString(r__));          \
    } while (0)

}  // namespace mb
