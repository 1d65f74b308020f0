// Fused NeRFSmall (HashNeRF tiny MLP) backward for sm_100a, the weight packing shared with the forward, the per-ray view term, and
// the C-ABI entry points of the NeRFSmall kernels.  The forward itself is mlp_small_fwd_tc_kernel (mlp_small_tc.cu).
//
// Replaces the autograd backward of NeRFSmallImpl::forward (reference src/NeRF.cpp:363-412: 5 cuBLAS SGEMMs + relu/slice/cat kernels,
// every [N,64] fp32 activation round-tripping HBM), including the keep-mask of RunNetwork (src/NeRFRenderer.h:187-188) and the
// per-sample direction expansion + SH + cat (:179-182).
//
//   sigma net : h0 = relu(enc32 · W0^T) ; d1 = h0 · W1^T          -> sigma = d1[:,0], geo = d1[:,1:16]
//   colour net: c  = relu(relu([sh16 | geo15] · W2^T) · W3^T) · W4^T
//   out [N,4] = [c0,c1,c2, sigma]                                   (src/NeRF.cpp:408; views first: :383)
//
// Activations are recomputed (nothing saved by the forward).  One warp owns 16 rows of a CTA tile and chains the five layers of the
// forward and then of the dX chain in registers: the fp32 accumulator fragment of one m16n8k16 mma.sync is re-packed (ReLU fused into
// the convert) as the A fragment of the next layer.  Weights live in shared memory pre-arranged in B-fragment order (nrf_mlp_small_pack),
// one conflict-free LDS.64 per MMA.  The forward runs fp16 x fp16 (the encodings ARE fp16 values, src/CuHashEmbedder.cu:253), the
// gradient chain bf16 x bf16; accumulation is fp32 throughout.  ReLU gates are kept as one 0xFFFF-per-active-half word per activation
// word (HSET2) and applied to the packed bf16 gradient pairs with a single AND; the next tile's inputs are requested at the start of the
// current one.  For dW = dY^T X, each warp drops its X_l / dY_l slabs into shared-memory tiles laid out as UMMA canonical MN-major
// regions; after one CTA barrier ONE thread issues 36 tcgen05.mma (SS form, both operands "K = rows"-major straight from those bytes)
// whose accumulators live in TMEM across the whole persistent loop, while the warps already work on the next tile; one fp32 atomicAdd
// per weight per CTA at the end.
//
// The A2 operand is laid out [sh(16) | d1(16)] instead of [sh(16) | geo(15) | pad]: column 16 is the sigma slot,
// whose weight column is zero (and whose value is zeroed), which avoids a cross-lane shift of the accumulators.
#include "mlp_small_layout.cuh"
#include "tcgen05.cuh"

namespace nrf {


__global__ void __launch_bounds__(256) mlp_pack_kernel(const float* __restrict__ p, int V, uint32_t* __restrict__ blob)
{
	const int w = blockIdx.x * blockDim.x + threadIdx.x;
	if (w >= kPackedWords) return;
	if (w >= kViewBase) {
		const int q = w - kViewBase, n = q >> 6, k = q & 63;
		reinterpret_cast<float*>(blob)[w] = k < V ? p[kW2 + n * w2_stride(V) + k] : 0.f;
		return;
	}
	if (w >= kUmmaBase) {
		// UMMA K-major core-matrix layout (mlp_small_layout.cuh): word q of layer l holds (n, k) and (n, k+1)
		int layer, base, N;
		if (w < kU1) { layer = 0; base = kU0; N = 64; }
		else if (w < kU2) { layer = 1; base = kU1; N = 16; }
		else if (w < kU3) { layer = 2; base = kU2; N = 64; }
		else if (w < kU4) { layer = 3; base = kU3; N = 64; }
		else { layer = 4; base = kU4; N = 16; }
		const auto [n, k] = tc::stage_word(w - base, N, 0);
		blob[w] = tc::pack_f16(wp(p, V, layer, n, k), wp(p, V, layer, n, k + 1));
		return;
	}
	int layer, base, NT;
	bool bwd = w >= kFwdWords;
	if (!bwd) {
		if (w < kF1) { layer = 0; base = kF0; NT = 8; }
		else if (w < kF2) { layer = 1; base = kF1; NT = 2; }
		else if (w < kF3) { layer = 2; base = kF2; NT = 8; }
		else if (w < kF4) { layer = 3; base = kF3; NT = 8; }
		else { layer = 4; base = kF4; NT = 1; }
	} else {
		if (w < kB3) { layer = 4; base = kB4; NT = 8; }
		else if (w < kB2) { layer = 3; base = kB3; NT = 8; }
		else if (w < kB1) { layer = 2; base = kB2; NT = 4; }
		else if (w < kB0) { layer = 1; base = kB1; NT = 8; }
		else { layer = 0; base = kB0; NT = 4; }
	}
	const int r = w - base;
	const int j = r & 1, lane = (r >> 1) & 31, tile = r >> 6;
	const int nt = tile % NT, ks = tile / NT;
	const int g = lane >> 2, t = lane & 3;
	const int nn = nt * 8 + g, kk = ks * 16 + 2 * t + 8 * j;
	float lo, hi;
	if (!bwd) {
		lo = wp(p, V, layer, nn, kk);
		hi = wp(p, V, layer, nn, kk + 1);
	} else {
		// B'[k'][n'] = Wp(k', n'): k' = output channel (padded with zero rows), n' = input channel
		const int n_out = layer == 1 ? 16 : (layer == 4 ? 8 : 64);
		lo = kk < n_out ? wp(p, V, layer, kk, nn) : 0.f;
		hi = kk + 1 < n_out ? wp(p, V, layer, kk + 1, nn) : 0.f;
	}
	// forward operands (activations AND weights) are fp16 on every layer: 10-bit mantissa, 8x fewer ReLU sign flips against
	// the fp32 reference than bf16; the gradient chain stays bf16 (fp32 range, no loss scale)
	blob[w] = !bwd ? tc::pack_f16(lo, hi) : tc::pack_bf16(lo, hi);
}

// ---------------------------------------------------------------------------------------------- MMA helpers
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
	asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
	             : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
	             : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
	asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
	             : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
	             : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// acc[NT][4] = A[KS] x frag  (frag: [ks][nt][lane] uint2 in shared memory)
template <int KS, int NT, bool F16>
__device__ __forceinline__ void layer_mma(const uint32_t (&a)[KS][4], const uint32_t* __restrict__ frag, int lane, float (&acc)[NT][4])
{
#pragma unroll
	for (int nt = 0; nt < NT; nt++) { acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f; }
	const uint2* f = reinterpret_cast<const uint2*>(frag);
#pragma unroll
	for (int ks = 0; ks < KS; ks++) {
#pragma unroll
		for (int nt = 0; nt < NT; nt++) {
			const uint2 b = f[(ks * NT + nt) * 32 + lane];
			if (F16) mma_f16(acc[nt], a[ks], b.x, b.y);
			else mma_bf16(acc[nt], a[ks], b.x, b.y);
		}
	}
}

// accumulator fragment of 2*KS n-tiles -> 16-bit A fragment of KS k-steps (F16: forward activations, else bf16 gradients)
template <int KS, bool RELU, bool F16>
__device__ __forceinline__ void repack(const float (&acc)[2 * KS][4], uint32_t (&a)[KS][4])
{
#pragma unroll
	for (int ks = 0; ks < KS; ks++) {
#pragma unroll
		for (int e = 0; e < 4; e++) {
			const float lo = acc[2 * ks + (e >> 1)][2 * (e & 1)], hi = acc[2 * ks + (e >> 1)][2 * (e & 1) + 1];
			a[ks][e] = F16 ? (RELU ? tc::pack_f16_relu(lo, hi) : tc::pack_f16(lo, hi)) : (RELU ? tc::pack_bf16_relu(lo, hi) : tc::pack_bf16(lo, hi));
		}
	}
}

// fp16 pair word -> bf16 pair word (the dW MMAs take bf16 x bf16: activations are re-quantised for that product only)
__device__ __forceinline__ uint32_t f16x2_to_bf16x2(uint32_t w)
{
	const float2 v = __half22float2(*reinterpret_cast<const __half2*>(&w));
	return tc::pack_bf16(v.x, v.y);
}
template <int KS>
__device__ __forceinline__ void to_bf16(const uint32_t (&a)[KS][4], uint32_t (&b)[KS][4])
{
#pragma unroll
	for (int ks = 0; ks < KS; ks++)
#pragma unroll
		for (int e = 0; e < 4; e++) b[ks][e] = f16x2_to_bf16x2(a[ks][e]);
}

// ---------------------------------------------------------------------------------------------- input loaders
// A fragment (fp16) of the 32 encoding channels for rows r_lo = row0+g, r_hi = row0+g+8.
template <int IN_KIND>
__device__ __forceinline__ void load_enc(const void* __restrict__ enc, int64_t r_lo, int64_t r_hi, int64_t n, int t, uint32_t (&a)[2][4])
{
	if (IN_KIND != NRF_MLP_IN_F32_CAT) {
		const uint32_t* e = reinterpret_cast<const uint32_t*>(enc);  // 16 words per row
#pragma unroll
		for (int ks = 0; ks < 2; ks++) {
			a[ks][0] = r_lo < n ? __ldg(e + r_lo * 16 + ks * 8 + t) : 0u;
			a[ks][1] = r_hi < n ? __ldg(e + r_hi * 16 + ks * 8 + t) : 0u;
			a[ks][2] = r_lo < n ? __ldg(e + r_lo * 16 + ks * 8 + 4 + t) : 0u;
			a[ks][3] = r_hi < n ? __ldg(e + r_hi * 16 + ks * 8 + 4 + t) : 0u;
		}
	} else {
		const float* x = reinterpret_cast<const float*>(enc);  // 48 floats per row
#pragma unroll
		for (int ks = 0; ks < 2; ks++) {
			float2 v;
			v = r_lo < n ? __ldg(reinterpret_cast<const float2*>(x + r_lo * 48 + ks * 16 + 2 * t)) : make_float2(0.f, 0.f);
			a[ks][0] = tc::pack_f16(v.x, v.y);
			v = r_hi < n ? __ldg(reinterpret_cast<const float2*>(x + r_hi * 48 + ks * 16 + 2 * t)) : make_float2(0.f, 0.f);
			a[ks][1] = tc::pack_f16(v.x, v.y);
			v = r_lo < n ? __ldg(reinterpret_cast<const float2*>(x + r_lo * 48 + ks * 16 + 8 + 2 * t)) : make_float2(0.f, 0.f);
			a[ks][2] = tc::pack_f16(v.x, v.y);
			v = r_hi < n ? __ldg(reinterpret_cast<const float2*>(x + r_hi * 48 + ks * 16 + 8 + 2 * t)) : make_float2(0.f, 0.f);
			a[ks][3] = tc::pack_f16(v.x, v.y);
		}
	}
}

// the four 8-byte loads of the 16 view channels (k-step 0 of the colour net input) of rows r_lo, r_hi, left un-converted (prefetch: a
// convert right after the load would stall on it)
template <int IN_KIND>
__device__ __forceinline__ void load_views_raw(const void* __restrict__ enc, const float* __restrict__ ray_sh, int S, int64_t r_lo, int64_t r_hi,
	int64_t n, int t, float2 (&v)[4])
{
	if (IN_KIND == NRF_MLP_IN_ENC16_RAYBIAS) {   // the view term arrives as a bias of the layer: k-step 0 of the colour input carries zeros
#pragma unroll
		for (int i = 0; i < 4; i++) v[i] = make_float2(0.f, 0.f);
		return;
	}
	const float* lo;
	const float* hi;
	if (IN_KIND == NRF_MLP_IN_ENC16_RAYDIRS) {
		lo = ray_sh + (r_lo < n ? r_lo / S : 0) * 16;
		hi = ray_sh + (r_hi < n ? r_hi / S : 0) * 16;
	} else {
		const float* x = reinterpret_cast<const float*>(enc);
		lo = x + (r_lo < n ? r_lo : 0) * 48 + 32;
		hi = x + (r_hi < n ? r_hi : 0) * 48 + 32;
	}
	v[0] = __ldg(reinterpret_cast<const float2*>(lo + 2 * t));
	v[1] = __ldg(reinterpret_cast<const float2*>(hi + 2 * t));
	v[2] = __ldg(reinterpret_cast<const float2*>(lo + 8 + 2 * t));
	v[3] = __ldg(reinterpret_cast<const float2*>(hi + 8 + 2 * t));
}

__device__ __forceinline__ void copy_blob(uint32_t* dst, const uint32_t* __restrict__ src, int words)
{
	const uint4* s = reinterpret_cast<const uint4*>(src);
	uint4* d = reinterpret_cast<uint4*>(dst);
	for (int i = threadIdx.x; i < words / 4; i += blockDim.x) d[i] = __ldg(s + i);
}

// ---------------------------------------------------------------------------------------------- backward
// 12 warps = 192 rows per CTA tile: three warps per scheduler to hide the latency of the dependent chain, at <= 170 registers per thread;
// the weights and the operand regions of a 192-row tile fill the shared memory one CTA may use
constexpr int kBwdWarps = 12;
constexpr int kBwdRows = kBwdWarps * 16;

// The X_l / dY_l tiles are stored as UMMA canonical MN-major regions [column chunk of 8][192 rows][8] bf16 (chunk stride 3072 B, 8-row
// group stride 128 B), so that dW = dY^T X is a handful of tcgen05.mma SS instructions per tile straight from these bytes (A and B both
// "rows = K"), accumulated in TMEM over the whole persistent loop.  Regions that share an MMA are adjacent: A operands are 128 columns
// wide (M = 128):
//   MMA1: A = [dY0 | dY2]  B = [X0 | X2] (N = 64)   -> rows 0..63 x cols 0..31 = dW0,  rows 64..127 x cols 32..63 = dW2
//   MMA2: A = [dY3 | X1 ]  B = [X3 | dY1] (N = 80)  -> rows 0..63 x cols 0..63 = dW3,  rows 64..127 x cols 64..79 = dW1^T
//   MMA3: A = [X4  | X3 ]  B = dY4 (N = 16)         -> rows 0..63 x cols 0..2  = dW4^T
// (the other quadrants are finite garbage that is never read back)
constexpr int kChunk = kBwdRows * 16;                          // bytes between 8-column chunks of a region
constexpr int kCRA = 0;                                        // [dY0 | dY2]
constexpr int kCRB = kCRA + kBwdRows * 128 * 2;                // [dY3 | X1]
constexpr int kCX4 = kCRB + kBwdRows * 128 * 2;
constexpr int kCX3 = kCX4 + kBwdRows * 64 * 2;
constexpr int kCD1 = kCX3 + kBwdRows * 64 * 2;
constexpr int kCX0 = kCD1 + kBwdRows * 16 * 2;
constexpr int kCX2 = kCX0 + kBwdRows * 32 * 2;
constexpr int kCD4 = kCX2 + kBwdRows * 32 * 2;
constexpr int kRegionBytes = kCD4 + kBwdRows * 16 * 2;         // 184 320
// weights + operand regions + the dW mbarrier and the TMEM address slot
constexpr size_t kBwdSmem = static_cast<size_t>(kBlobWords) * 4 + kRegionBytes + 64;
constexpr uint32_t kDwT0 = 0, kDwT1 = 64, kDwT2 = 144;        // TMEM columns of the three accumulators

// store an A-fragment-shaped register set (KS k-steps) for rows (g, g+8) of this warp's slab into a region, from 8-column chunk chunk0 on
template <int KS, int CHUNK>
__device__ __forceinline__ void store_frag_c(uint8_t* region, int chunk0, int row_g, int t, const uint32_t (&a)[KS][4])
{
	uint8_t* p = region + chunk0 * CHUNK + row_g * 16 + t * 4;
#pragma unroll
	for (int ks = 0; ks < KS; ks++) {
		*reinterpret_cast<uint32_t*>(p + (2 * ks) * CHUNK) = a[ks][0];
		*reinterpret_cast<uint32_t*>(p + (2 * ks) * CHUNK + 128) = a[ks][1];          // row + 8
		*reinterpret_cast<uint32_t*>(p + (2 * ks + 1) * CHUNK) = a[ks][2];
		*reinterpret_cast<uint32_t*>(p + (2 * ks + 1) * CHUNK + 128) = a[ks][3];
	}
}

// per-element ReLU gates of an activation fragment: 0xFFFF where the fp16 activation is > 0 (one HSET2 per word); the gradient
// fragment of the same layer has the same (k-step, element) layout, so gating is one AND per packed bf16 pair
template <int KS>
__device__ __forceinline__ void relu_gates(const uint32_t (&a)[KS][4], uint32_t (&m)[KS][4])
{
	const __half2 zero = __float2half2_rn(0.f);
#pragma unroll
	for (int ks = 0; ks < KS; ks++)
#pragma unroll
		for (int e = 0; e < 4; e++) m[ks][e] = __hgt2_mask(*reinterpret_cast<const __half2*>(&a[ks][e]), zero);
}
template <int KS>
__device__ __forceinline__ void apply_gates(uint32_t (&d)[KS][4], const uint32_t (&m)[KS][4])
{
#pragma unroll
	for (int ks = 0; ks < KS; ks++)
#pragma unroll
		for (int e = 0; e < 4; e++) d[ks][e] &= m[ks][e];
}

// NRF_MLP_IN_ENC16_RAYBIAS: acc (colour layer 0 pre-activation, [8 n-tiles][4]) += bias[ray of the row][64]
__device__ __forceinline__ void add_ray_bias(float (&acc)[8][4], const float* __restrict__ bias, int S, int64_t r_lo, int64_t r_hi, int64_t n, int t)
{
	const float* lo = bias + (r_lo < n ? r_lo / S : 0) * 64 + 2 * t;
	const float* hi = bias + (r_hi < n ? r_hi / S : 0) * 64 + 2 * t;
#pragma unroll
	for (int nt = 0; nt < 8; nt++) {
		const float2 a = __ldg(reinterpret_cast<const float2*>(lo + nt * 8)), b = __ldg(reinterpret_cast<const float2*>(hi + nt * 8));
		acc[nt][0] += a.x; acc[nt][1] += a.y; acc[nt][2] += b.x; acc[nt][3] += b.y;
	}
}

// NRF_MLP_IN_ENC16_RAYBIAS: grad_bias[ray][64] += column sums of the slab's gated bf16 gradient of that pre-activation (A-fragment layout).
// The 16 rows of a slab belong to ONE ray (samples_per_ray is a multiple of 16, host-checked; rows past n carry zeros).
__device__ __forceinline__ void reduce_ray_bias_grad(const uint32_t (&d)[4][4], float* __restrict__ grad_bias, int S, int64_t slab_row0, int64_t n, int g, int t)
{
	float2 s[8];
#pragma unroll
	for (int ks = 0; ks < 4; ks++)
#pragma unroll
		for (int h = 0; h < 2; h++) {
			const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&d[ks][2 * h]));
			const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&d[ks][2 * h + 1]));
			s[2 * ks + h] = make_float2(a.x + b.x, a.y + b.y);
		}
#pragma unroll
	for (int off = 4; off < 32; off <<= 1)
#pragma unroll
		for (int i = 0; i < 8; i++) {
			s[i].x += __shfl_xor_sync(0xffffffffu, s[i].x, off);
			s[i].y += __shfl_xor_sync(0xffffffffu, s[i].y, off);
		}
	if (g == 0 && slab_row0 < n) {
		float* o = grad_bias + (slab_row0 / S) * 64 + 2 * t;
#pragma unroll
		for (int i = 0; i < 8; i++) {          // columns 8 i + 2 t, + 1
			if (s[i].x != 0.f) atomicAdd(o + 8 * i, s[i].x);
			if (s[i].y != 0.f) atomicAdd(o + 8 * i + 1, s[i].y);
		}
	}
}

template <int IN_KIND>
__global__ void __launch_bounds__(kBwdWarps * 32, 1) mlp_small_bwd_kernel(const uint32_t* __restrict__ blob, const void* __restrict__ enc,
	const float* __restrict__ ray_sh, int S, const uint8_t* __restrict__ keep, int64_t n, const float* __restrict__ grad_raw,
	void* __restrict__ grad_in, float* __restrict__ grad_params, int V, float* __restrict__ grad_bias)
{
	extern __shared__ __align__(16) uint8_t smem_raw[];
	uint32_t* wf = reinterpret_cast<uint32_t*>(smem_raw);
	uint8_t* ctiles = smem_raw + static_cast<size_t>(kBlobWords) * 4;                       // the operand regions
	uint64_t* dw_done = reinterpret_cast<uint64_t*>(ctiles + kRegionBytes);                 // the tile's MMAs have read the regions
	uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ctiles + kRegionBytes + 8);
	const int lane = threadIdx.x & 31, warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), g = lane >> 2, t = lane & 3;
	if (warp == 0) {
		if (lane == 0) {
			tc::mbar_init(dw_done, 1);
			asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		}
		__syncwarp();
		tc::tmem_alloc_all(tmem_slot);
	}
	copy_blob(wf, blob, kBlobWords);
	tc::fence_before();
	__syncthreads();
	tc::fence_after();
	const uint32_t tmem = *tmem_slot;
	const int row_g = warp * 16 + g;  // row inside the CTA tile

	uint32_t it = 0;                  // tiles done by this CTA

	const int64_t n_tiles = (n + kBwdRows - 1) / kBwdRows;
	// inputs of the tile in flight (prefetched one tile ahead)
	uint32_t in_a0[2][4];
	float2 in_v[4];
	float4 in_g_lo, in_g_hi;
	uint8_t in_k_lo = 1, in_k_hi = 1;
	auto load_tile = [&](int64_t tile) {   // loads only: every consumer of the loaded values sits in the next iteration
		const int64_t r_lo = tile * kBwdRows + row_g, r_hi = r_lo + 8;
		load_enc<IN_KIND>(enc, r_lo, r_hi, n, t, in_a0);
		load_views_raw<IN_KIND>(enc, ray_sh, S, r_lo, r_hi, n, t, in_v);
		in_g_lo = make_float4(0.f, 0.f, 0.f, 0.f);
		in_g_hi = in_g_lo;
		if (r_lo < n) in_g_lo = __ldg(reinterpret_cast<const float4*>(grad_raw + r_lo * 4));
		if (r_hi < n) in_g_hi = __ldg(reinterpret_cast<const float4*>(grad_raw + r_hi * 4));
		in_k_lo = (keep && r_lo < n) ? __ldg(keep + r_lo) : uint8_t(1);
		in_k_hi = (keep && r_hi < n) ? __ldg(keep + r_hi) : uint8_t(1);
	};
	if (static_cast<int64_t>(blockIdx.x) < n_tiles) load_tile(blockIdx.x);
	for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
		const int64_t r_lo = tile * kBwdRows + row_g, r_hi = r_lo + 8;
		float4 g_lo = in_g_lo, g_hi = in_g_hi;
		if (!in_k_lo) g_lo.w = 0.f;               // d(sigma) is dropped outside the box (src/NeRFRenderer.h:188)
		if (!in_k_hi) g_hi.w = 0.f;
		uint32_t cur_a0[2][4];
		float2 cur_v[4];
#pragma unroll
		for (int ks = 0; ks < 2; ks++)
#pragma unroll
			for (int e = 0; e < 4; e++) cur_a0[ks][e] = in_a0[ks][e];
#pragma unroll
		for (int e = 0; e < 4; e++) cur_v[e] = in_v[e];
		// the weight-gradient MMAs are issued by one thread and the warps loop straight on, so the next tile's inputs are requested HERE, a whole
		// recompute + gradient chain ahead of their first use
		if (tile + gridDim.x < n_tiles) load_tile(tile + gridDim.x);
		uint32_t m1[4][4], m3[4][4], m4[4][4];   // ReLU gates of X1, X3, X4
		// ---- forward recompute; every layer input is dropped into its X region (bf16, packed straight from the fp32 accumulators)
		{
			uint32_t a0[2][4];
#pragma unroll
			for (int ks = 0; ks < 2; ks++)
#pragma unroll
				for (int e = 0; e < 4; e++) a0[ks][e] = cur_a0[ks][e];
			float acc[8][4];
			layer_mma<2, 8, true>(a0, wf + kF0, lane, acc);
			uint32_t xb2[2][4], xb4[4][4];                               // bf16 copies for the dW products
			to_bf16<2>(a0, xb2);
			// the previous tile's weight-gradient MMAs must be done with the regions before the first store into them (they ran behind layer 0)
			if (it > 0) tc::mbar_wait(dw_done, (it - 1) & 1u);
			store_frag_c<2, kChunk>(ctiles + kCX0, 0, row_g, t, xb2);
			uint32_t a1[4][4];
			repack<4, true, true>(acc, a1);
			relu_gates<4>(a1, m1);
			repack<4, true, false>(acc, xb4);
			store_frag_c<4, kChunk>(ctiles + kCRB, 8, row_g, t, xb4);
			float d1[2][4];
			layer_mma<4, 2, true>(a1, wf + kF1, lane, d1);
			uint32_t a2[2][4];
#pragma unroll
			for (int e = 0; e < 4; e++) a2[0][e] = tc::pack_f16(cur_v[e].x, cur_v[e].y);
			if (t == 0) { d1[0][0] = 0.f; d1[0][2] = 0.f; }
			repack<1, false, true>(d1, reinterpret_cast<uint32_t(&)[1][4]>(a2[1]));
			to_bf16<2>(a2, xb2);
			store_frag_c<2, kChunk>(ctiles + kCX2, 0, row_g, t, xb2);
			layer_mma<2, 8, true>(a2, wf + kF2, lane, acc);
			if (IN_KIND == NRF_MLP_IN_ENC16_RAYBIAS) add_ray_bias(acc, ray_sh, S, r_lo, r_hi, n, t);
			uint32_t a3[4][4];
			repack<4, true, true>(acc, a3);
			relu_gates<4>(a3, m3);
			repack<4, true, false>(acc, xb4);
			store_frag_c<4, kChunk>(ctiles + kCX3, 0, row_g, t, xb4);
			layer_mma<4, 8, true>(a3, wf + kF3, lane, acc);
			repack<4, true, true>(acc, a3);
			relu_gates<4>(a3, m4);
			repack<4, true, false>(acc, xb4);
			store_frag_c<4, kChunk>(ctiles + kCX4, 0, row_g, t, xb4);
		}
		// ---- backward chain
		{
			uint32_t d4[1][4];
			d4[0][0] = t == 0 ? tc::pack_bf16(g_lo.x, g_lo.y) : (t == 1 ? tc::pack_bf16(g_lo.z, 0.f) : 0u);
			d4[0][1] = t == 0 ? tc::pack_bf16(g_hi.x, g_hi.y) : (t == 1 ? tc::pack_bf16(g_hi.z, 0.f) : 0u);
			d4[0][2] = 0u;
			d4[0][3] = 0u;
			store_frag_c<1, kChunk>(ctiles + kCD4, 0, row_g, t, d4);         // 8 real + 8 zero columns
			float acc[8][4];
			layer_mma<1, 8, false>(d4, wf + kB4, lane, acc);                 // dA4 = dD4 · W4
			uint32_t d3[4][4];
			repack<4, false, false>(acc, d3);
			apply_gates<4>(d3, m4);
			store_frag_c<4, kChunk>(ctiles + kCRB, 0, row_g, t, d3);
			layer_mma<4, 8, false>(d3, wf + kB3, lane, acc);                 // dA3 = dD3 · W3
			repack<4, false, false>(acc, d3);
			apply_gates<4>(d3, m3);
			if (IN_KIND == NRF_MLP_IN_ENC16_RAYBIAS) reduce_ray_bias_grad(d3, grad_bias, S, tile * kBwdRows + warp * 16, n, g, t);
			store_frag_c<4, kChunk>(ctiles + kCRA, 8, row_g, t, d3);
			float da2[4][4];
			layer_mma<4, 4, false>(d3, wf + kB2, lane, da2);                 // dA2 = dD2 · W2p  (cols 0..15 views, 16..31 d1)
			if (t == 0) { da2[2][0] += g_lo.w; da2[2][2] += g_hi.w; }        // + d(sigma)
			uint32_t dd1[1][4];
			dd1[0][0] = tc::pack_bf16(da2[2][0], da2[2][1]);
			dd1[0][1] = tc::pack_bf16(da2[2][2], da2[2][3]);
			dd1[0][2] = tc::pack_bf16(da2[3][0], da2[3][1]);
			dd1[0][3] = tc::pack_bf16(da2[3][2], da2[3][3]);
			store_frag_c<1, kChunk>(ctiles + kCD1, 0, row_g, t, dd1);
			layer_mma<1, 8, false>(dd1, wf + kB1, lane, acc);                // dA1 = dD1 · W1
			repack<4, false, false>(acc, d3);
			apply_gates<4>(d3, m1);
			store_frag_c<4, kChunk>(ctiles + kCRA, 0, row_g, t, d3);
			if (grad_in) {
				float de[4][4];
				layer_mma<4, 4, false>(d3, wf + kB0, lane, de);             // dEnc = dD0 · W0
				if (IN_KIND != NRF_MLP_IN_F32_CAT) {
					uint32_t* o = reinterpret_cast<uint32_t*>(grad_in);      // bf16 [N,32] = 16 words per row
#pragma unroll
					for (int nt = 0; nt < 4; nt++) {
						if (r_lo < n) o[r_lo * 16 + nt * 4 + t] = tc::pack_bf16(de[nt][0], de[nt][1]);
						if (r_hi < n) o[r_hi * 16 + nt * 4 + t] = tc::pack_bf16(de[nt][2], de[nt][3]);
					}
				} else {
					float* o = reinterpret_cast<float*>(grad_in);            // fp32 [N,48]
#pragma unroll
					for (int nt = 0; nt < 4; nt++) {
						if (r_lo < n) *reinterpret_cast<float2*>(o + r_lo * 48 + nt * 8 + 2 * t) = make_float2(de[nt][0], de[nt][1]);
						if (r_hi < n) *reinterpret_cast<float2*>(o + r_hi * 48 + nt * 8 + 2 * t) = make_float2(de[nt][2], de[nt][3]);
					}
#pragma unroll
					for (int nt = 0; nt < 2; nt++) {
						if (r_lo < n) *reinterpret_cast<float2*>(o + r_lo * 48 + 32 + nt * 8 + 2 * t) = make_float2(da2[nt][0], da2[nt][1]);
						if (r_hi < n) *reinterpret_cast<float2*>(o + r_hi * 48 + 32 + nt * 8 + 2 * t) = make_float2(da2[nt][2], da2[nt][3]);
					}
				}
			}
		}
		// ---- dW on tcgen05: 3 MMAs per 16-row K step straight from the regions, accumulators stay in TMEM
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");          // the st.shared above -> visible to the MMA's async reads
		__syncthreads();
		if (warp == 0) {
			const uint32_t base = tc::smem_u32(ctiles);
			const uint64_t a1 = tc::smem_desc(base + kCRA, 128, kChunk), b1 = tc::smem_desc(base + kCX0, 128, kChunk);
			const uint64_t a2 = tc::smem_desc(base + kCRB, 128, kChunk), b2 = tc::smem_desc(base + kCX3, 128, kChunk);
			const uint64_t a3 = tc::smem_desc(base + kCX4, 128, kChunk), b3 = tc::smem_desc(base + kCD4, 128, kChunk);
			const uint32_t first = it ? 1u : 0u;
			if (tc::elect_one()) {
				tc::fence_after();
#pragma unroll
				for (int j = 0; j < kBwdWarps; j++) {                            // K = 16 rows per step: +256 B on both descriptors
					const uint64_t o = static_cast<uint64_t>(16 * j);
					tc::umma_ss(tmem + kDwT0, a1 + o, b1 + o, tc::idesc(128, 64, true, 1, 1), j ? 1u : first);
					tc::umma_ss(tmem + kDwT1, a2 + o, b2 + o, tc::idesc(128, 80, true, 1, 1), j ? 1u : first);
					tc::umma_ss(tmem + kDwT2, a3 + o, b3 + o, tc::idesc(128, 16, true, 1, 1), j ? 1u : first);
				}
				tc::umma_commit(dw_done);
			}
			__syncwarp();
		}
		it++;
	}

	// ---- flush: one thread per accumulator row (TMEM lane), fp32 atomics into the flat gradient
	if (it > 0) tc::mbar_wait(dw_done, (it - 1) & 1u);
	tc::fence_after();
	if (warp < 4 && it > 0) {
		const int m = warp * 32 + lane;
		const uint32_t t_lane = tmem + (static_cast<uint32_t>(warp * 32) << 16);
		for (int c0 = 0; c0 < 160; c0 += 16) {
			uint32_t d16[16];
			tc::tmem_ld16(t_lane + c0, d16);
			tc::tmem_ld_wait();
#pragma unroll
			for (int j = 0; j < 16; j++) {
				const int c = c0 + j;
				int idx = -1;
				if (c < 64) idx = (m < 64) ? (c < 32 ? w_index(V, 0, m, c) : -1) : (c >= 32 ? w_index(V, 2, m - 64, c - 32) : -1);
				else if (c < 144) idx = (m < 64) ? (c < 128 ? w_index(V, 3, m, c - 64) : -1) : (c >= 128 ? w_index(V, 1, c - 128, m - 64) : -1);
				else idx = (m < 64) ? w_index(V, 4, c - 144, m) : -1;
				const float v = __uint_as_float(d16[j]);
				if (idx >= 0 && v != 0.f) atomicAdd(grad_params + idx, v);
			}
		}
	}
	tc::fence_before();
	__syncthreads();
	if (warp == 0) {
		tc::fence_after();
		tc::tmem_free_all(tmem);
	}
}

// ---------------------------------------------------------------------------------------------- per-ray view term (NRF_MLP_IN_ENC16_RAYBIAS)
// bias[r][n] = sum_k ray_sh[r][k] W2[n][k], k < V, in fp32 (the one place the view channels meet their weights: once per RAY, not per sample).
// One CTA stages the view block of W2 (64 x V floats) and walks kRaysPerBlock rays, 64 outputs each.  Optionally zeroes the grad_bias rows of its
// rays (the accumulator reduce_ray_bias_grad adds into later in the step).
constexpr int kViewBiasThreads = 256, kRaysPerBlock = 16;

__global__ void __launch_bounds__(kViewBiasThreads) view_bias_fwd_kernel(const uint32_t* __restrict__ blob, int V, const float* __restrict__ ray_sh, int64_t R,
	float* __restrict__ bias, float* __restrict__ grad_bias_zero)
{
	extern __shared__ float vb_smem[];
	float* w = vb_smem;                              // [64][V + 1]
	float* sh = vb_smem + 64 * (V + 1);              // [4][V]
	for (int i = threadIdx.x; i < 64 * V; i += blockDim.x) {
		const int n = i / V, k = i - n * V;
		w[n * (V + 1) + k] = reinterpret_cast<const float*>(blob)[kViewBase + n * 64 + k];
	}
	const int n = threadIdx.x & 63, q = threadIdx.x >> 6;
	const int64_t ray0 = static_cast<int64_t>(blockIdx.x) * kRaysPerBlock;
	for (int pass = 0; pass < kRaysPerBlock / 4; pass++) {
		__syncthreads();
		const int64_t rbase = ray0 + pass * 4;
		for (int i = threadIdx.x; i < 4 * V; i += blockDim.x) {
			const int64_t r = rbase + i / V;
			sh[i] = r < R ? ray_sh[r * V + (i % V)] : 0.f;
		}
		__syncthreads();
		const int64_t r = rbase + q;
		if (r < R) {
			float acc = 0.f;
			for (int k = 0; k < V; k++) acc = fmaf(sh[q * V + k], w[n * (V + 1) + k], acc);
			bias[r * 64 + n] = acc;
			if (grad_bias_zero) grad_bias_zero[r * 64 + n] = 0.f;
		}
	}
}

// dW2[n][k] += sum_r grad_bias[r][n] ray_sh[r][k], k < V.  A CTA reduces kBiasBwdRays rays from shared memory; thread = (n, 16 consecutive k / 4).
constexpr int kBiasBwdRays = 64;

__global__ void __launch_bounds__(256) view_bias_bwd_kernel(const float* __restrict__ ray_sh, int V, const float* __restrict__ grad_bias, int64_t R,
	float* __restrict__ grad_params)
{
	extern __shared__ float vb_smem[];
	float* g = vb_smem;                              // [kBiasBwdRays][64]
	float* sh = vb_smem + kBiasBwdRays * 64;         // [kBiasBwdRays][V]
	const int64_t ray0 = static_cast<int64_t>(blockIdx.x) * kBiasBwdRays;
	for (int i = threadIdx.x; i < kBiasBwdRays * 64; i += blockDim.x) {
		const int64_t r = ray0 + i / 64;
		g[i] = r < R ? grad_bias[r * 64 + (i & 63)] : 0.f;
	}
	for (int i = threadIdx.x; i < kBiasBwdRays * V; i += blockDim.x) {
		const int64_t r = ray0 + i / V;
		sh[i] = r < R ? ray_sh[r * V + (i % V)] : 0.f;
	}
	__syncthreads();
	for (int o = threadIdx.x; o < 64 * V; o += blockDim.x) {
		const int n = o / V, k = o - n * V;
		float acc = 0.f;
		for (int r = 0; r < kBiasBwdRays; r++) acc = fmaf(g[r * 64 + n], sh[r * V + k], acc);
		if (acc != 0.f) atomicAdd(grad_params + kW2 + n * w2_stride(V) + k, acc);
	}
}

// mlp_small_tc.cu
cudaError_t launch_mlp_small_fwd_tc(const uint32_t* blob, int in_kind, const void* enc, const float* ray_sh, int S, const uint8_t* keep, int64_t n,
	float* raw_out, cudaStream_t stream);
cudaError_t launch_mlp_small_fwd_tc_importance(const uint32_t* blob, int in_kind, const void* enc, const float* ray_sh, const uint8_t* keep, const int16_t* perm,
	int64_t n_rays, int n_importance, int n_merged, float* raw_out, cudaStream_t stream);

static int check_shape(const nrf_mlp_small_shape* s)
{
	NRF_REQUIRE(s != nullptr, "shape is null");
	if (!(s->input_ch == 32 && s->input_ch_views >= 1 && s->input_ch_views <= 64 && s->hidden_dim == 64 && s->geo_feat_dim == 15 &&
	      s->hidden_dim_color == 64 && s->num_layers == 2 && s->num_layers_color == 3)) {
		set_error("nrf_mlp_small: built for 32 + V -> 64 -> 16 | V + 15 -> 64 -> 64 -> 3 with 1 <= V <= 64 view channels (SH degree 1..8)");
		return NRF_ERR_UNSUPPORTED;
	}
	return NRF_OK;
}

// the per-sample view input (k-step 0 of the colour net) exists for V = 16 only; other V go through the per-ray bias
static int check_in_kind(const nrf_mlp_small_shape* s, nrf_mlp_input in_kind)
{
	NRF_REQUIRE(in_kind == NRF_MLP_IN_ENC16_RAYDIRS || in_kind == NRF_MLP_IN_F32_CAT || in_kind == NRF_MLP_IN_ENC16_RAYBIAS, "bad in_kind");
	if (s->input_ch_views != 16 && in_kind != NRF_MLP_IN_ENC16_RAYBIAS) {
		set_error("nrf_mlp_small: input_ch_views != 16 runs as NRF_MLP_IN_ENC16_RAYBIAS (nrf_mlp_small_view_bias_fwd / _bwd carry the view term)");
		return NRF_ERR_UNSUPPORTED;
	}
	return NRF_OK;
}

}  // namespace nrf

using namespace nrf;

extern "C" {

int64_t nrf_mlp_small_packed_bytes(const nrf_mlp_small_shape* shape) { return check_shape(shape) ? -1 : static_cast<int64_t>(kPackedWords) * 4; }
int64_t nrf_mlp_small_param_count(const nrf_mlp_small_shape* shape) { return check_shape(shape) ? -1 : param_count(shape->input_ch_views); }

int nrf_mlp_small_pack(const nrf_mlp_small_shape* shape, const float* params_flat, void* packed, nrf_stream stream)
{
	if (int rc = check_shape(shape)) return rc;
	NRF_REQUIRE(params_flat && packed, "null pointer");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 15) == 0, "packed blob must be 16-byte aligned");
	mlp_pack_kernel<<<(kPackedWords + 255) / 256, 256, 0, as_stream(stream)>>>(params_flat, shape->input_ch_views, reinterpret_cast<uint32_t*>(packed));
	NRF_CHECK_LAUNCH("mlp_pack_kernel");
	return NRF_OK;
}

int nrf_mlp_small_view_bias_fwd(const nrf_mlp_small_shape* shape, const void* packed, const float* ray_sh, int64_t n_rays, float* bias_out,
	float* grad_bias_zero, nrf_stream stream)
{
	if (int rc = check_shape(shape)) return rc;
	NRF_REQUIRE(n_rays >= 0, "negative n_rays");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(packed && ray_sh && bias_out, "null pointer");
	const int V = shape->input_ch_views;
	const size_t smem = static_cast<size_t>(64 * (V + 1) + 4 * V) * sizeof(float);
	const unsigned blocks = static_cast<unsigned>((n_rays + kRaysPerBlock - 1) / kRaysPerBlock);
	view_bias_fwd_kernel<<<blocks, kViewBiasThreads, smem, as_stream(stream)>>>(reinterpret_cast<const uint32_t*>(packed), V, ray_sh, n_rays, bias_out,
		grad_bias_zero);
	NRF_CHECK_LAUNCH("view_bias_fwd_kernel");
	return NRF_OK;
}

int nrf_mlp_small_view_bias_bwd(const nrf_mlp_small_shape* shape, const float* ray_sh, const float* grad_bias, int64_t n_rays, float* grad_params_flat,
	nrf_stream stream)
{
	if (int rc = check_shape(shape)) return rc;
	NRF_REQUIRE(n_rays >= 0, "negative n_rays");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(ray_sh && grad_bias && grad_params_flat, "null pointer");
	const int V = shape->input_ch_views;
	const size_t smem = static_cast<size_t>(kBiasBwdRays) * (64 + V) * sizeof(float);
	const unsigned blocks = static_cast<unsigned>((n_rays + kBiasBwdRays - 1) / kBiasBwdRays);
	view_bias_bwd_kernel<<<blocks, 256, smem, as_stream(stream)>>>(ray_sh, V, grad_bias, n_rays, grad_params_flat);
	NRF_CHECK_LAUNCH("view_bias_bwd_kernel");
	return NRF_OK;
}

int nrf_mlp_small_fwd(const nrf_mlp_small_shape* shape, const void* packed, nrf_mlp_input in_kind, const void* enc,
	const float* ray_sh, int32_t samples_per_ray, const uint8_t* keep, int64_t n, float* raw_out, nrf_stream stream)
{
	if (int rc = check_shape(shape)) return rc;
	if (int rc = check_in_kind(shape, in_kind)) return rc;
	NRF_REQUIRE(n >= 0, "negative n");
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(packed && enc && raw_out, "null pointer");
	NRF_REQUIRE(in_kind == NRF_MLP_IN_F32_CAT || (ray_sh && samples_per_ray >= 1), "ray_sh / samples_per_ray missing");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 15) == 0, "packed blob must be 16-byte aligned");
	NRF_REQUIRE(in_kind == NRF_MLP_IN_F32_CAT || (reinterpret_cast<uintptr_t>(enc) & 15) == 0, "enc must be 16-byte aligned");
	NRF_CUDA(launch_mlp_small_fwd_tc(reinterpret_cast<const uint32_t*>(packed), in_kind, enc, ray_sh, samples_per_ray, keep, n, raw_out,
		as_stream(stream)));
	count_launch();
	return NRF_OK;
}

int nrf_mlp_small_fwd_importance(const nrf_mlp_small_shape* shape, const void* packed, nrf_mlp_input in_kind, const void* enc_merged, const float* ray_sh,
	const uint8_t* keep_merged, const int16_t* perm, int64_t n_rays, int32_t n_importance, int32_t n_merged, float* raw_merged, nrf_stream stream)
{
	if (int rc = check_shape(shape)) return rc;
	if (int rc = check_in_kind(shape, in_kind)) return rc;
	NRF_REQUIRE(in_kind != NRF_MLP_IN_F32_CAT, "the importance-only forward reads fp16 encodings (RAYDIRS / RAYBIAS)");
	NRF_REQUIRE(n_rays >= 0 && n_importance >= 1 && n_merged > n_importance && n_merged < 32768, "bad sizes");
	NRF_REQUIRE(n_rays * n_merged < (int64_t(1) << 31), "n_rays * n_merged must be < 2^31 per call");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(packed && enc_merged && ray_sh && perm && raw_merged, "null pointer");
	NRF_REQUIRE(((reinterpret_cast<uintptr_t>(packed) | reinterpret_cast<uintptr_t>(enc_merged) | reinterpret_cast<uintptr_t>(raw_merged)) & 15) == 0,
		"packed / enc_merged / raw_merged must be 16-byte aligned");
	NRF_CUDA(launch_mlp_small_fwd_tc_importance(reinterpret_cast<const uint32_t*>(packed), in_kind, enc_merged, ray_sh, keep_merged, perm, n_rays, n_importance,
		n_merged, raw_merged, as_stream(stream)));
	count_launch();
	return NRF_OK;
}

int nrf_mlp_small_bwd(const nrf_mlp_small_shape* shape, const void* packed, nrf_mlp_input in_kind, const void* enc,
	const float* ray_sh, int32_t samples_per_ray, const uint8_t* keep, int64_t n, const float* grad_raw, void* grad_in,
	float* grad_params_flat, nrf_stream stream)
{
	NRF_REQUIRE(in_kind != NRF_MLP_IN_ENC16_RAYBIAS, "NRF_MLP_IN_ENC16_RAYBIAS: use nrf_mlp_small_bwd_raybias (it also returns the gradient of the bias)");
	return nrf_mlp_small_bwd_raybias(shape, packed, in_kind, enc, ray_sh, samples_per_ray, keep, n, grad_raw, grad_in, grad_params_flat, nullptr, stream);
}

int nrf_mlp_small_bwd_raybias(const nrf_mlp_small_shape* shape, const void* packed, nrf_mlp_input in_kind, const void* enc,
	const float* ray_sh, int32_t samples_per_ray, const uint8_t* keep, int64_t n, const float* grad_raw, void* grad_in,
	float* grad_params_flat, float* grad_bias, nrf_stream stream)
{
	if (int rc = check_shape(shape)) return rc;
	if (int rc = check_in_kind(shape, in_kind)) return rc;
	NRF_REQUIRE(n >= 0, "negative n");
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(packed && enc && grad_raw && grad_params_flat, "null pointer");
	NRF_REQUIRE(in_kind == NRF_MLP_IN_F32_CAT || (ray_sh && samples_per_ray >= 1), "ray_sh / samples_per_ray missing");
	NRF_REQUIRE(in_kind != NRF_MLP_IN_ENC16_RAYBIAS || (grad_bias && samples_per_ray % 16 == 0),
		"NRF_MLP_IN_ENC16_RAYBIAS needs grad_bias and samples_per_ray % 16 == 0 (a 16-row slab must lie within one ray)");
	const int V = shape->input_ch_views;
	const uint32_t* blob = reinterpret_cast<const uint32_t*>(packed);
	const int blocks = static_cast<int>(std::min<int64_t>((n + kBwdRows - 1) / kBwdRows, kNumSMs));
	auto kernel = mlp_small_bwd_kernel<NRF_MLP_IN_F32_CAT>;
	if (in_kind == NRF_MLP_IN_ENC16_RAYDIRS) kernel = mlp_small_bwd_kernel<NRF_MLP_IN_ENC16_RAYDIRS>;
	else if (in_kind == NRF_MLP_IN_ENC16_RAYBIAS) kernel = mlp_small_bwd_kernel<NRF_MLP_IN_ENC16_RAYBIAS>;
	NRF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kBwdSmem)));
	kernel<<<blocks, kBwdWarps * 32, kBwdSmem, as_stream(stream)>>>(blob, enc, ray_sh, samples_per_ray, keep, n, grad_raw, grad_in,
		grad_params_flat, V, grad_bias);
	NRF_CHECK_LAUNCH("mlp_small_bwd_kernel");
	return NRF_OK;
}

}
