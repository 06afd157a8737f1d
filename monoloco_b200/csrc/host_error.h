// Host-side error reporting shared by every C-ABI entry point: the message goes to the thread-local text that
// mlb_last_error() returns, and the entry point returns -1.
#pragma once
#include <cuda_runtime.h>

#include <string>

extern thread_local std::string g_mlb_err;
void mlb_count_launch();  // one kernel launch issued (mlb_launch_count)

inline int mlb_fail(const std::string& msg) {
    g_mlb_err = msg;
    return -1;
}

// cudaMalloc + zero fill
template <class T>
cudaError_t mlb_zalloc(T** ptr, size_t bytes) {
    const cudaError_t e = cudaMalloc(ptr, bytes);
    return e != cudaSuccess ? e : cudaMemset(*ptr, 0, bytes);
}

#define MLB_CU(call)                                                                                  \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess) return mlb_fail(std::string(#call) + ": " + cudaGetErrorString(e_));  \
    } while (0)
