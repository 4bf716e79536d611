// okp_common.cuh -- shared device helpers for libokp.so (sm_100a).
//
// Arithmetic contract (kept identical to oracle/np_oracle.py and oracle/okp_oracle.c):
// the library is compiled with -fmad=false so every float/double product and sum is rounded
// separately, exactly like the reference's NumPy / torch-CPU arithmetic.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../include/okp.h"

#define OKP_CUDA_CHECK(expr)                         \
    do {                                             \
        cudaError_t _e = (expr);                     \
        if (_e != cudaSuccess) return OKP_E_CUDA;    \
    } while (0)

// One candidate peak as the tile kernels hand it to the merge step (32 bytes).
struct OkpPeakRecord {
    int32_t key;     // y * W + x: raster order
    float score;     // box sum at the peak
    float cx, cy;    // centroid (x, y)
    float conf;      // sum of the window's probabilities
    int32_t pad[3];
};

struct OkpConfig { int32_t cfg[OKP_MAX_MAPS]; };    // cfg[0] = 1 (centre map), then keypoint_config

__device__ __forceinline__ int okp_min(int a, int b) { return a < b ? a : b; }
__device__ __forceinline__ int okp_max(int a, int b) { return a > b ? a : b; }
__device__ __forceinline__ int okp_clamp(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Map element types. float32 is the reference's type; bfloat16 is what a bf16 network head writes
// (BASELINE config 5); float16 is what torch.autocast on CUDA, model.half() or a half-precision TorchScript
// export writes. bf16 -> f32 and f16 -> f32 are exact (every float16, subnormals included, is a float32
// value), so every kernel computes on the very float32 values the oracle sees when it is handed the up-cast
// map: the parity contract does not change with the type.
template <typename T> __device__ __forceinline__ float okp_ld(const T* p);
template <> __device__ __forceinline__ float okp_ld<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float okp_ld<__nv_bfloat16>(const __nv_bfloat16* p) {
    return __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p)) << 16);
}
template <> __device__ __forceinline__ float okp_ld<__half>(const __half* p) { return __half2float(__ldg(p)); }

// Programmatic dependent launch (sm_90+): a kernel launched with okp_launch_dependent() may be scheduled while the kernel
// in front of it on the stream drains -- its launch latency (2-4 us between dependent kernels on a B200) overlaps the
// predecessor's tail. It must call okp_wait_for_predecessor() before it touches anything the predecessor wrote; the wait
// returns when the predecessor grid has completed and its writes are visible (a no-op under an ordinary launch).
__device__ __forceinline__ void okp_wait_for_predecessor() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... KernelArgs, typename... Args>
static inline cudaError_t okp_launch_dependent(void (*kernel)(KernelArgs...), dim3 grid, dim3 block, size_t smem,
                                               cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t config;
    memset(&config, 0, sizeof(config));
    config.gridDim = grid; config.blockDim = block; config.dynamicSmemBytes = smem; config.stream = stream;
    cudaLaunchAttribute attribute;
    attribute.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attribute.val.programmaticStreamSerializationAllowed = 1;
    config.attrs = &attribute; config.numAttrs = 1;
    return cudaLaunchKernelEx(&config, kernel, KernelArgs(args)...);
}
