// common.h -- host-side helpers shared by the translation units of libdfb_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>

#include "dfb_require.h"

namespace dfb {
int check_cuda(cudaError_t e, const char* what);
}  // namespace dfb

#define DFB_CUDA(call)                                   \
    do {                                                 \
        int _r = dfb::check_cuda((call), #call);         \
        if (_r != DFB_OK) return _r;                     \
    } while (0)

#define DFB_LAUNCH_CHECK(name)                                        \
    do {                                                              \
        int _r = dfb::check_cuda(cudaGetLastError(), "launch " name); \
        if (_r != DFB_OK) return _r;                                  \
    } while (0)
