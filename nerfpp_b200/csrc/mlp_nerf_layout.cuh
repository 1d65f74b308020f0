// Layer tables, packed-weight blob and activation / gradient scratch layouts shared by the fused classic-NeRF kernels
// (mlp_nerf_tc.cu: forward, inference and training; mlp_nerf_bwd_tc.cu: gradient chain and weight gradients).
//
// Packed weights (nrf_mlp_nerf_pack / _pack_train): layer l travels as stages of 64 input columns; inside a stage element
// (n = output, k = input) sits at byte (k/8)*(N*16) + n*16 + (k%8)*2, i.e. 8 x 16-byte UMMA core matrices.  The SAME bytes are
//   * a K-major   B operand with MN = outputs, K = inputs  (forward:  D[rows, out] = A[rows, in]  * W^T), SBO 128, LBO N*16
//   * an MN-major B operand with MN = inputs,  K = outputs (backward: D[rows, in]  = dY[rows, out] * W ), SBO N*16, LBO 128
// so the gradient chain streams the forward blob and only the descriptors change.
//
// Activation / gradient scratch (training): one record per 128-row tile, made of regions of C columns stored as
// [row half (2)][C/8 column chunks][64 rows][8 elements] bf16.  A 64-row half of any 128-column range is contiguous, and is at
// the same time the MN-major A operand (M = columns, K = rows) and the MN-major B operand (N = columns, K = rows) of the weight-
// gradient product dW = dY^T X, with SBO 1024 (column chunks) and LBO 128 (8-row groups): the producers write 16-byte chunks
// per row (512 contiguous bytes per warp instruction) and the consumer needs ONE bulk copy per operand and stage.
#pragma once
#include "tcgen05.cuh"

namespace nrf {
namespace nerf_tc {

using namespace tc;

constexpr int kW = 256, kInPts = 63, kInViews = 27, kInCh = kInPts + kInViews;

// TMEM columns of the forward kernel
constexpr uint32_t kColD = 0, kColD16 = 256, kColPts = 272, kColH = 304, kColViews = 432;

// id: 0..7 pts_linears, 8 feature_linear, 9 alpha_linear, 10 views_linears[0], 11 rgb_linear
constexpr int kLayers = 12;
struct LayerInfo {
	int N, K;            // padded
	uint32_t a_col, d_col;
};
__host__ __device__ constexpr LayerInfo layer_info(int l)
{
	return l == 0 ? LayerInfo{256, 64, kColPts, kColD}
	     : l == 5 ? LayerInfo{256, 320, kColPts, kColD}
	     : l <= 8 ? LayerInfo{256, 256, kColH, kColD}
	     : l == 9 ? LayerInfo{16, 256, kColH, kColD16}
	     : l == 10 ? LayerInfo{128, 288, kColH, kColD}
	     : LayerInfo{16, 128, kColH, kColD16};
}
// the narrow heads (N = 16) travel as ONE stage holding their whole K; everything else in 64-wide K slabs (last one may be 32)
__host__ __device__ constexpr int layer_stages(int l) { return layer_info(l).N == 16 ? 1 : (layer_info(l).K + 63) / 64; }
__host__ __device__ constexpr int stage_k(int l, int s)
{
	return layer_info(l).N == 16 ? layer_info(l).K : (layer_info(l).K - 64 * s >= 64 ? 64 : layer_info(l).K - 64 * s);
}
__host__ __device__ constexpr int stage_bytes(int l, int s) { return layer_info(l).N * stage_k(l, s) * 2; }
__host__ __device__ constexpr int layer_bytes(int l)
{
	int b = 0;
	for (int s = 0; s < layer_stages(l); s++) b += stage_bytes(l, s);
	return b;
}
__host__ __device__ constexpr int layer_offset(int l)
{
	int b = 0;
	for (int i = 0; i < l; i++) b += layer_bytes(i);
	return b;
}
__host__ __device__ constexpr int stage_offset(int l, int s)
{
	int b = layer_offset(l);
	for (int i = 0; i < s; i++) b += stage_bytes(l, i);
	return b;
}
constexpr int kWeightBytes = layer_offset(kLayers);
// biases (fp32) follow the weights: [layer][N padded]
__host__ __device__ constexpr int bias_offset(int l)
{
	int b = 0;
	for (int i = 0; i < l; i++) b += layer_info(i).N;
	return b;
}
constexpr int kBiasFloats = bias_offset(kLayers);
constexpr int kPackedBytes = kWeightBytes + kBiasFloats * 4;
constexpr int kRing = 4;
constexpr int kStageBytes = 256 * 64 * 2;       // largest stage: N = 256, K = 64

// ---- training scratch: per-tile records (region_bytes / chunk_offset: tcgen05.cuh) ------------------------------------
// saved activations (operands of the weight-gradient products): pts(64) views(32) h1..h8 (256 each: h_l = input of pts_linears[l]; h8 feeds feature / alpha) feature(256) hv(128)
constexpr int kSavePts = 0;
constexpr int kSaveViews = kSavePts + region_bytes(64);
__host__ __device__ constexpr int save_h(int l) { return kSaveViews + region_bytes(32) + (l - 1) * region_bytes(256); }
constexpr int kSaveFeat = save_h(9);
constexpr int kSaveHv = kSaveFeat + region_bytes(256);
// ReLU masks, one bit per unit, for the gradient chain (which then never reads the activations themselves): 9 sets per tile
// (0: hv, l = 1..8: h_l), each [128 rows][8 words]; word c of a row covers columns 32c .. 32c+31, bit i = column 32c + 2i,
// bit 16 + i = column 32c + 2i + 1 (the low / high halves of the i-th packed bf16 pair: two instructions per pair to build)
constexpr int kSaveBits = kSaveHv + region_bytes(128);
__host__ __device__ constexpr int bits_offset(int set, int row) { return kSaveBits + set * 4096 + row * 32; }
constexpr int kSaveTile = kSaveBits + 9 * 4096;                 // 684 032 B per 128 rows
// gradients of the pre-activations: dOut(16: [r,g,b,alpha,0..]) d_hv(128) d_feature(256) dY_0..dY_7 (256 each)
constexpr int kGradOut = 0;
constexpr int kGradHv = kGradOut + region_bytes(16);
constexpr int kGradFeat = kGradHv + region_bytes(128);
__host__ __device__ constexpr int grad_y(int l) { return kGradFeat + region_bytes(256) + l * region_bytes(256); }
constexpr int kGradTile = grad_y(8);                            // 626 688 B per 128 rows

struct Weights {   // device pointers, torch Linear layout [out, in] row-major fp32
	const float* w[kLayers];
	const float* b[kLayers];
};
struct Grads {     // same order, accumulated into (+=)
	float* w[kLayers];
	float* b[kLayers];
};

int check_shape(const nrf_mlp_nerf_shape* s);

}  // namespace nerf_tc
}  // namespace nrf
