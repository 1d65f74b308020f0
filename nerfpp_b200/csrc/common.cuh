// Shared helpers for the sm_100a kernels behind include/nerfpp_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/nerfpp_b200.h"

namespace nrf {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

inline cudaStream_t as_stream(nrf_stream s) { return reinterpret_cast<cudaStream_t>(s); }

// launch check: never synchronises, only picks up launch-configuration errors
#define NRF_CHECK_LAUNCH(what)                                                          \
	do {                                                                                \
		cudaError_t e__ = cudaGetLastError();                                           \
		if (e__ != cudaSuccess) {                                                       \
			nrf::set_error("%s: %s", what, cudaGetErrorString(e__));                    \
			return NRF_ERR_CUDA;                                                        \
		}                                                                               \
		nrf::count_launch();                                                            \
	} while (0)

#define NRF_CUDA(call)                                                                  \
	do {                                                                                \
		cudaError_t e__ = (call);                                                       \
		if (e__ != cudaSuccess) {                                                       \
			nrf::set_error("%s: %s", #call, cudaGetErrorString(e__));                   \
			return NRF_ERR_CUDA;                                                        \
		}                                                                               \
	} while (0)

#define NRF_REQUIRE(cond, msg)                                                          \
	do {                                                                                \
		if (!(cond)) {                                                                  \
			nrf::set_error("%s: %s", __func__, msg);                                    \
			return NRF_ERR_INVALID;                                                     \
		}                                                                               \
	} while (0)

constexpr int kNumSMs = 148;  // B200

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
	return v;
}

// inclusive prefix sum across the warp
__device__ __forceinline__ float warp_scan_incl(float v, int lane)
{
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) {
		float n = __shfl_up_sync(0xffffffffu, v, o);
		if (lane >= o) v += n;
	}
	return v;
}

// inclusive suffix sum across the warp (lane i gets sum over lanes >= i)
__device__ __forceinline__ float warp_scan_incl_rev(float v, int lane)
{
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) {
		float n = __shfl_down_sync(0xffffffffu, v, o);
		if (lane + o < 32) v += n;
	}
	return v;
}

}  // namespace nrf
