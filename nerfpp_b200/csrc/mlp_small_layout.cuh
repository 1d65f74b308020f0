// Packed-weight blob of the fused NeRFSmall kernels (nrf_mlp_small_pack): layout constants shared by the mma.sync backward
// (mlp_small.cu) and the tcgen05 forward (mlp_small_tc.cu).
//
//   words [0, kFwdWords)            forward B fragments for mma.sync m16n8k16 (the backward's recompute), fp16, [layer][ks][nt][lane][2]
//   words [kFwdWords, kBlobWords)   backward (transposed) B fragments, bf16
//   words [kViewBase, kPackedWords) fp32 view block of colour layer 0 for the per-ray view term (NRF_MLP_IN_ENC16_RAYBIAS)
//   words [kUmmaBase, kTotalWords)  forward weights as UMMA shared-memory operands (tcgen05.mma B, K-major, no swizzle), fp16:
//                                   layer l at kU<l>; element (n, k) at byte (k/8)*(N*16) + n*16 + (k%8)*2, i.e. 8x16-byte
//                                   core matrices with SBO = 128 B between 8-row groups and LBO = N*16 B between K chunks
#pragma once
#include "common.cuh"

namespace nrf {

constexpr int kW0 = 0, kW1 = 2048, kW2 = 3072, kW3 = 5056, kW4 = 9152, kParamCount = 9344;  // flat fp32 offsets
// fragment blob, offsets in 32-bit words.  fwd: [ks][nt][lane][2]
constexpr int kF0 = 0, kF1 = 1024, kF2 = 1536, kF3 = 2560, kF4 = 4608, kFwdWords = 4864;
constexpr int kB4 = 4864, kB3 = 5376, kB2 = 7424, kB1 = 8448, kB0 = 8960, kBlobWords = 9984;

// V = input_ch_views.  The kernels are built around 16 view channels as k-step 0 of the colour net's first layer; any other V (SH degree != 4:
// 64 at the reference's shipped degree 8, src/main.cpp:176) takes the per-ray form NRF_MLP_IN_ENC16_RAYBIAS — the view term views . W2[:, :V]^T
// depends on the RAY only, so it is computed once per ray (view_bias kernels) and enters the fused kernels as a bias of that layer, whose k-step
// 0 then carries zeros.  Flat fp32 layout for any V: W2 is [64, V + 15] and the layers after it move by 64 (V - 16).
__host__ __device__ constexpr int w2_stride(int V) { return V + 15; }
__host__ __device__ constexpr int off_w3(int V) { return kW2 + 64 * (V + 15); }
__host__ __device__ constexpr int off_w4(int V) { return off_w3(V) + 64 * 64; }
__host__ __device__ constexpr int param_count(int V) { return off_w4(V) + 3 * 64; }
static_assert(off_w3(16) == kW3 && off_w4(16) == kW4 && param_count(16) == kParamCount, "V = 16 is the built-in layout");

// flat index of padded element (layer, out n, padded in k), -1 for padding.  Layer 2's padded input is [views(16) | sigma slot | geo(15)];
// with V != 16 its view columns belong to the per-ray term and are not part of the padded matrix.
__host__ __device__ __forceinline__ int w_index(int V, int layer, int n, int k)
{
	switch (layer) {
		case 0: return kW0 + n * 32 + k;
		case 1: return kW1 + n * 64 + k;
		case 2: return k < 16 ? (V == 16 ? kW2 + n * 31 + k : -1) : (k == 16 ? -1 : kW2 + n * w2_stride(V) + V + k - 17);
		case 3: return off_w3(V) + n * 64 + k;
		default: return n < 3 ? off_w4(V) + n * 64 + k : -1;
	}
}

// padded logical weight matrices Wp_l(n, k)
__device__ __forceinline__ float wp(const float* __restrict__ p, int V, int layer, int n, int k)
{
	const int i = w_index(V, layer, n, k);
	return i >= 0 ? p[i] : 0.f;
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi)
{
	__nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
	return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi)
{
	__half2 v = __floats2half2_rn(lo, hi);
	return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_bf16_relu(float lo, float hi)
{
	uint32_t r;
	asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
	return r;
}


__device__ __forceinline__ uint32_t pack_f16_relu(float lo, float hi)
{
	uint32_t r;
	asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
	return r;
}

// UMMA operand region (fp16), offsets in 32-bit words; padded N: layer 1 -> 16, layer 4 -> 16 (rows 3..15 zero)
constexpr int kUmmaBase = kBlobWords;
constexpr int kU0 = kUmmaBase, kU1 = kU0 + 64 * 32 / 2, kU2 = kU1 + 16 * 64 / 2, kU3 = kU2 + 64 * 32 / 2, kU4 = kU3 + 64 * 64 / 2;
constexpr int kTotalWords = kU4 + 16 * 64 / 2;
constexpr int kUmmaWords = kTotalWords - kUmmaBase;   // 5120 words = 20 KiB
// fp32 copy of the view block of the colour net's first layer, [64][64] (column k < V real, the rest zero): what the per-ray view term
// (view_bias_fwd_kernel) multiplies with — so that inference needs nothing but the blob
constexpr int kViewBase = kTotalWords;
constexpr int kPackedWords = kViewBase + 64 * 64;

}  // namespace nrf
