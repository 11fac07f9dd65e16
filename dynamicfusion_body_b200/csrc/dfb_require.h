// dfb_require.h -- argument checks of the C ABI (include/dfb.h).  Plain C++ (no CUDA runtime) so that the host-side set-up of
// every entry point runs unchanged in the library and in the test suite's host build.
#pragma once
#include "../../include/dfb.h"

namespace dfb {

void set_error(const char* fmt, ...);  // provided by common.cu (library) or the test suite's host build

}  // namespace dfb

#define DFB_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            dfb::set_error(__VA_ARGS__);  \
            return DFB_ERR_INVALID;       \
        }                                 \
    } while (0)
