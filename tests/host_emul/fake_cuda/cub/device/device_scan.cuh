// TEST INFRASTRUCTURE ONLY -- stand-in for cub::DeviceScan::ExclusiveSum under the SIMT emulator.
#pragma once
#include <cuda_runtime.h>
namespace cub {
struct DeviceScan {
    template <typename In, typename Out, typename N>
    static cudaError_t ExclusiveSum(void* temp, size_t& temp_bytes, const In* in, Out* out, N n, cudaStream_t = nullptr) {
        if (!temp) { temp_bytes = 16; return cudaSuccess; }
        Out acc = Out(0);
        for (N i = 0; i < n; ++i) {
            const Out v = (Out)in[i];
            out[i] = acc;
            acc += v;
        }
        return cudaSuccess;
    }
};
}  // namespace cub
