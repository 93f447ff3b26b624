// Internal helpers shared by the libdctd translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/dctd.h"

namespace dctd {

void set_cuda_error(cudaError_t e);   // records into the thread-local "last CUDA error", clears the runtime's pending one
void count_launch(int n = 1);         // bumps the thread-local launch counter

#define DCTD_CUDA_TRY(expr)                      \
    do {                                         \
        cudaError_t _e = (expr);                 \
        if (_e != cudaSuccess) {                 \
            ::dctd::set_cuda_error(_e);          \
            return DCTD_ERR_CUDA;                \
        }                                        \
    } while (0)

#define DCTD_LAUNCH_CHECK()                      \
    do {                                         \
        cudaError_t _e = cudaGetLastError();     \
        if (_e != cudaSuccess) {                 \
            ::dctd::set_cuda_error(_e);          \
            return DCTD_ERR_CUDA;                \
        }                                        \
        ::dctd::count_launch();                  \
    } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace dctd
