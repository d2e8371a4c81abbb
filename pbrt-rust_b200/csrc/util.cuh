// CUDA error plumbing.
#pragma once
#include <cuda_runtime.h>
#include <string>
#include "error.h"
#include "../../include/pbrt_b200.h"

#define PB_CUDA_TRY(call)                                                                              \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) {                                                                      \
            cudaGetLastError();                                                                        \
            return pbrt_b200::fail(e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver     \
                                       ? PBRT_B200_ERR_NO_DEVICE : PBRT_B200_ERR_CUDA,                \
                                   std::string(#call) + ": " + cudaGetErrorString(e__));               \
        }                                                                                              \
    } while (0)

using pbrt_b200::fail;
