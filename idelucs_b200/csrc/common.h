// idelucs_b200 — internal helpers shared by the .cu translation units.
#pragma once
#include <cuda_runtime.h>

#include "../../include/idelucs_b200.h"

namespace idl {
// records the thread-local error text returned by idl_last_error(); returns `code`
int set_error(int code, const char* fmt, const char* a = "", long long b = 0);
// counts the kernels this library has launched (idl_launch_count)
void note_launch();
// IDL_EINVAL naming `who` unless 0 <= row_begin <= row_end <= n (hdbscan.cu; the row ranges of the all-pairs entry points)
int check_rows(const char* who, int64_t n, int64_t row_begin, int64_t row_end);
}  // namespace idl

#define IDL_CUDA_CHECK(expr)                                                                             \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            return ::idl::set_error(IDL_ECUDA, "%s (cuda error %lld)", cudaGetErrorString(_e), (long long)_e); \
    } while (0)
