// Layer tables, operand blob and training-record layouts shared by the fused LeRF language-head kernels
// (lerf_tc.cu: forward programs; lerf_bwd_tc.cu: gradient chain, weight gradients, per-ray backward) — SURVEY §8f-1, BASELINE C5.
//
//   sigma net   h1 = relu(W_s0 x)  [256]      s = W_s1 h1  [33] = [sigma_le | geo_feat 32]                 (reference src/LeRF.cpp:86-93)
//   language    h2 = relu(W_e0 [geo | x])  [256]      e = W_e1 h2  [512]      out = [e / max(|e|, 1e-8) | sigma_le]      (:96-110)
//
// Operand blob (nrf_lerf_pack): layer l travels as stages of 64 input columns; inside a stage element (n = output, k = input) sits at byte
// (k/8)*(N*16) + n*16 + (k%8)*2, i.e. 8 x 16-byte UMMA core matrices.  The SAME bytes are
//   * a K-major   B operand with MN = outputs, K = inputs  (forward:  D[rows, out] = A[rows, in]  * W^T), SBO 128, LBO N*16
//   * an MN-major B operand with MN = inputs,  K = outputs (backward: D[rows, in]  = dY[rows, out] * W ), SBO N*16, LBO 128
// so the gradient chain streams the forward blob and only the descriptors change (the mlp_nerf_layout.cuh scheme).
// Two copies: fp16 (the forward programs SIGMA / HIDDEN / RAW / TRAIN and the chain's G h2 product: activations are O(1) and keep 11 bits)
// and bf16 (the gradient products of the chain: gradient rows need fp32's exponent range).  A and B of one tcgen05.mma kind::f16 must share
// their 16-bit format (a mixed descriptor faults on B200), so the weight-gradient products dW = dY^T X read BF16 copies of the activations.
#pragma once
#include "tcgen05.cuh"

namespace nrf {
namespace lerf_tc {

using namespace tc;

constexpr int kIn = 128, kHid = 256, kGeo = 32, kDim = 512, kSigN = 48;   // kSigN: the 33 outputs of the sigma head padded to a UMMA N
constexpr uint32_t kColD = 0, kColD2 = 256, kColGeo = 304, kColEnc = 320, kColH = 384;
constexpr int kRing = 4;
constexpr int kStageBytes = 256 * 64 * 2;

// layers: 0 S0 (128 -> 256), 1 S1 (256 -> [geo 32 | sigma | 0..]), 2 E0 (160 -> 256), 3 G (256 -> 256), 4 / 5 E1 outputs 0..255 / 256..511
constexpr int kLayers = 6;
struct LayerInfo {
	int N, K;
	uint32_t a_col, d_col;
};
__host__ __device__ constexpr LayerInfo layer_info(int l)
{
	return l == 0 ? LayerInfo{kHid, kIn, kColEnc, kColD}
	     : l == 1 ? LayerInfo{kSigN, kHid, kColH, kColD2}
	     : l == 2 ? LayerInfo{kHid, kGeo + kIn, kColGeo, kColD}
	              : LayerInfo{kHid, kHid, kColH, kColD};
}
// the narrow sigma head travels as ONE stage holding its whole K (24 KB); everything else in 64-wide K slabs (E0's last one is 32)
__host__ __device__ constexpr int layer_stages(int l) { return l == 1 ? 1 : (layer_info(l).K + 63) / 64; }
__host__ __device__ constexpr int stage_k(int l, int s) { return l == 1 ? layer_info(l).K : (layer_info(l).K - 64 * s >= 64 ? 64 : layer_info(l).K - 64 * s); }
__host__ __device__ constexpr int stage_bytes(int l, int s) { return layer_info(l).N * stage_k(l, s) * 2; }
__host__ __device__ constexpr int layer_bytes(int l) { return layer_info(l).N * layer_info(l).K * 2; }
__host__ __device__ constexpr int layer_offset(int l)
{
	int b = 0;
	for (int i = 0; i < l; i++) b += layer_bytes(i);
	return b;
}
constexpr int kWeightBytes = layer_offset(kLayers);             // 565 248: the fp16 copy of all six layers
// the bf16 copy of S0, S1, E0 (+ G, unused) for the gradient chain, same per-layer sizes / offsets; W_e0's input columns reordered [x | geo]
constexpr int kTrainBase = kWeightBytes;
constexpr int kTrainBytes = layer_offset(4);                    // 303 104
// W_e1 transposed, fp32 [256 k][512 n], follows the operand blobs (lerf_project_kernel reads it)
constexpr int kProjBase = kTrainBase + kTrainBytes;
constexpr int kProjBytes = kHid * kDim * 4;
// one fp32 after it: the power-of-two scale the 16-bit copies of G were divided by (lerf_gscale_kernel), so that a trained W_e1 cannot overflow fp16
constexpr int kScaleBase = kProjBase + kProjBytes;
// and G = W_e1^T W_e1 itself in fp32 [256][256] (lerf_gram_kernel; the pack kernel rounds the 16-bit operand copies from it)
constexpr int kGramBase = kScaleBase + 128;
constexpr int kPackedBytes = kGramBase + kHid * kHid * 4;
static_assert(kWeightBytes % 128 == 0 && kTrainBytes % 128 == 0, "blob alignment");

// stage programs: the weight stages one 128-row tile consumes, in order, as (byte offset in the blob, bytes)
enum Mode { kSigma = 0, kHidden = 1, kRaw = 2, kTrain = 3, kChain = 4 };
constexpr int kModes = 5;
struct ModeTable {
	int n_groups, group_layer[8];
	int n_stages, off[24], bytes[24];
};
constexpr ModeTable make_mode(int mode)
{
	ModeTable t{};
	const int seq_sigma[2] = {0, 1}, seq_hidden[4] = {0, 1, 2, 3}, seq_raw[7] = {0, 1, 2, 4, 5, 4, 5}, seq_chain[4] = {3, 2, 1, 0};
	t.n_groups = mode == kSigma ? 2 : (mode == kRaw ? 7 : 4);
	for (int g = 0; g < t.n_groups; g++)
		t.group_layer[g] = mode == kSigma ? seq_sigma[g] : (mode == kRaw ? seq_raw[g] : (mode == kChain ? seq_chain[g] : seq_hidden[g]));
	int i = 0;
	for (int g = 0; g < t.n_groups; g++) {
		const int l = t.group_layer[g];
		// the chain reads G from the fp16 copy (its A operand h2 is fp16) and W_e0, W_s1, W_s0 from the bf16 copy (A operand = bf16 gradient rows)
		int off = ((mode == kChain && l != 3) ? kTrainBase : 0) + layer_offset(l);
		for (int s = 0; s < layer_stages(l); s++, i++) {
			t.off[i] = off;
			t.bytes[i] = stage_bytes(l, s);
			off += stage_bytes(l, s);
		}
	}
	t.n_stages = i;
	return t;
}
static_assert(make_mode(kSigma).n_stages == 3 && make_mode(kHidden).n_stages == 10 && make_mode(kRaw).n_stages == 22 && make_mode(kChain).n_stages == 10,
	"stage programs");

// h2 tile records of the HIDDEN program (inference): [32 column chunks][128 rows][8 fp16] = 64 KB per 128-row tile; a warp store covers 512 contiguous bytes
constexpr int kHiddenTile = 128 * kHid * 2;

// ---- training records, one per 128-row tile, made of regions of C columns in the record layout of tcgen05.cuh (region_bytes / chunk_offset):
// a 64-row half of a region is the MN-major A or B operand of a weight-gradient product dW = dY^T X.
// saved by the training forward: bf16 copies of [geo 32 | x 128] (the input of le_net[0]), h1 and h2 (B / A operands of the weight-gradient
// products), h2 once more in fp16 (what the forward itself multiplied: the A operand of the chain's G h2 product and the source of the per-ray
// sums, whose rounding the density gradient — a cancellation-prone residual of the compositing backward — amplifies), and the ReLU mask of h1
// (one bit per unit: word c of a row covers columns 32c .. 32c+31, bit i = column 32c + 2i, bit 16 + i = column 32c + 2i + 1 — the low / high
// halves of the i-th packed pair)
constexpr int kSaveGX = 0;
constexpr int kSaveH1 = kSaveGX + region_bytes(kGeo + kIn);
constexpr int kSaveH2 = kSaveH1 + region_bytes(kHid);             // fp16
constexpr int kSaveH2B = kSaveH2 + region_bytes(kHid);            // bf16
constexpr int kSaveBits1 = kSaveH2B + region_bytes(kHid);
constexpr int kSaveTile = kSaveBits1 + 128 * 32;                 // 241 664 B per 128 rows
// written by the gradient chain (bf16): d a2 (256), d s = [d geo 32 | d sigma | 0..] (48), d a1 (256), beta * h2 (256: A operand of the weighted Gram matrix)
constexpr int kGradA2 = 0;
constexpr int kGradS = kGradA2 + region_bytes(kHid);
constexpr int kGradA1 = kGradS + region_bytes(kSigN);
constexpr int kGradBH2 = kGradA1 + region_bytes(kHid);
constexpr int kGradTile = kGradBH2 + region_bytes(kHid);         // 208 896 B per 128 rows

__device__ __forceinline__ float2 half2_bits_to_float2(uint32_t w) { return __half22float2(*reinterpret_cast<const __half2*>(&w)); }
__device__ __forceinline__ uint32_t half2_bits_to_bf16x2(uint32_t w)
{
	const float2 f = half2_bits_to_float2(w);
	return pack_bf16(f.x, f.y);
}

struct Weights {   // device pointers, torch Linear layout [out, in] row-major fp32, no biases (src/LeRF.cpp:12,15)
	const float* s0;   // [256, 128]
	const float* s1;   // [33, 256]   row 0 = sigma_le, rows 1..32 = geo_feat_le (src/LeRF.cpp:92-93)
	const float* e0;   // [256, 160]  columns [geo 32 | enc 128] (src/LeRF.cpp:96)
	const float* e1;   // [512, 256]
};

int check_shape(const nrf_lerf_shape* s);

}  // namespace lerf_tc
}  // namespace nrf
