// Fused NeRFSmall forward on the 5th-generation tensor cores (tcgen05 / TMEM / TMA) for sm_100a.
//
// NeRFSmallImpl::forward (reference src/NeRF.cpp:363-412), the per-sample direction expansion + SH + cat and the keep-mask write
// (src/NeRFRenderer.h:179-188); the packing, the backward and the C-ABI entry points are in mlp_small.cu.  Machine mapping:
//   * a CTA owns the SM (persistent, 1 CTA/SM) and all 512 TMEM columns, split into kSlots independent tile pipelines;
//   * each pipeline processes 128 sample points at a time: M = 128 rows = the 128 TMEM lanes, one epilogue thread per row;
//   * every layer is tcgen05.mma.cta_group::1.kind::f16 with M=128, N=64 (or 16), K=16 per instruction:
//         A  (activations)  lives in TENSOR MEMORY  (written by the epilogue threads with tcgen05.st, fp16 pairs per column)
//         B  (weights)      lives in SHARED MEMORY  (K-major core matrices, staged once per CTA by one TMA bulk copy)
//         D  (accumulator)  lives in TENSOR MEMORY  (fp32, read back with tcgen05.ld)
//     so the chain enc -> h0 -> [sigma|geo] -> colour net never touches shared or global memory between layers;
//   * every pipeline has its own issuing thread (lane 0 of its first epilogue warp): it waits for the pipeline's "A ready"
//     mbarrier (one arrival per epilogue warp), issues the layer's 2-4 MMAs with compile-time descriptors and signals
//     "D ready" with tcgen05.commit.  The tensor pipe works on one pipeline while the others run their epilogues
//     (ReLU + fp16 pack + tcgen05.st) — the epilogue round trip, not the MMA, is the long pole of a 64-wide MLP.
//     (r1c profile: ONE thread issuing for all four pipelines spent ~730 cycles of dependent scalar work per layer step
//     and capped the tensor pipe at 10 %; profiles/r1_mlp_small_fwd_tc_v1_ncu.txt.)
//   * the next tile's encodings are loaded while the current tile runs its last two layers.
//
// TMEM columns of pipeline s (base = 128 s):  [0,64) D of the 64-wide layers | [64,80) D of the 16-wide layers |
//                                             [96,128) A operand of the next layer (K <= 64 fp16 = 32 columns)
#include "mlp_small_layout.cuh"
#include "tcgen05.cuh"

namespace nrf {

namespace tc {

constexpr int kSlots = 4;                    // tile pipelines per CTA (4 x 128 TMEM columns)
constexpr int kThreads = 128 * kSlots;     // 4 epilogue warps per pipeline; lane 0 of each pipeline's first warp issues its MMAs
constexpr uint32_t kColD = 0, kColD16 = 64, kColA = 96, kSlotCols = 128;

// compile-time description of layer L: offset in the staged blob (words), padded out channels N, K/16, accumulator column
template <int L> struct Layer;
template <> struct Layer<0> { static constexpr int off = kU0 - kUmmaBase, N = 64, KS = 2; static constexpr uint32_t d_col = kColD; };
template <> struct Layer<1> { static constexpr int off = kU1 - kUmmaBase, N = 16, KS = 4; static constexpr uint32_t d_col = kColD16; };
template <> struct Layer<2> { static constexpr int off = kU2 - kUmmaBase, N = 64, KS = 2; static constexpr uint32_t d_col = kColD; };
template <> struct Layer<3> { static constexpr int off = kU3 - kUmmaBase, N = 64, KS = 4; static constexpr uint32_t d_col = kColD; };
template <> struct Layer<4> { static constexpr int off = kU4 - kUmmaBase, N = 16, KS = 4; static constexpr uint32_t d_col = kColD16; };

struct __align__(16) Smem {
	uint32_t w[kUmmaWords];            // 20 KiB of UMMA B operands
	uint64_t w_ready;
	uint64_t a_ready[kSlots];          // 4 epilogue warps -> the slot's issuing thread
	uint64_t d_ready[kSlots];          // tcgen05.commit -> epilogue threads
	uint32_t tmem_base;
};

// 32 fp32 accumulator columns -> 16 fp16-pair words, ReLU fused into the convert
__device__ __forceinline__ void relu_pack(const uint32_t (&acc)[32], uint32_t (&out)[16])
{
#pragma unroll
	for (int i = 0; i < 16; i++) out[i] = pack_f16_relu(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1]));
}

// The slot's issuing thread: wait until the four epilogue warps have published the A operand, issue the K/16 MMAs of
// layer L (every descriptor field is a compile-time constant but the two base addresses), commit to d_ready.
template <int L>
__device__ __forceinline__ void issue_layer(uint64_t* a_ready, uint64_t* d_ready, uint32_t& pa, uint32_t col, uint32_t w_saddr)
{
	using LY = Layer<L>;
	constexpr uint32_t id = idesc(128, LY::N, false, 0, 0);
	constexpr uint32_t lbo = LY::N * 16;   // bytes between the two 8-wide K chunks of one instruction
	mbar_wait(a_ready, pa);
	pa ^= 1u;
	fence_after();
#pragma unroll
	for (int j = 0; j < LY::KS; j++) {
		const uint64_t bd = smem_desc(w_saddr + LY::off * 4 + j * 2 * lbo, lbo, 128);
		umma_ts(col + LY::d_col, col + kColA + j * 8, bd, id, j > 0);
	}
	umma_commit(d_ready);
}

struct RowInputs {
	uint32_t e[16];   // layer-0 operand: the row's 32 fp16 encodings
	uint32_t v[8];    // the row's 16 view channels as fp16 pairs (layer-2 operand, K chunk 0)
	bool kept;
};

// Importance-only evaluation (nrf_mlp_small_fwd_importance): work row r = (ray, j < N) lives at row ray * T + perm[ray, j] of the
// merged fine-pass arrays (perm: nrf_sample_pdf_merge_perm); perm == nullptr: rows are their own positions.
struct RowMap {
	const int16_t* perm;
	int N, T;
};

__device__ __forceinline__ int64_t merged_row(const RowMap& m, int64_t r, int64_t n)
{
	if (r >= n) return 0;
	const uint32_t ray = static_cast<uint32_t>(r) / static_cast<uint32_t>(m.N);
	const uint32_t j = static_cast<uint32_t>(r) - ray * static_cast<uint32_t>(m.N);
	const int64_t row0 = static_cast<int64_t>(ray) * m.T;
	return row0 + m.perm[row0 + j];
}

// r: the row's position in enc / keep / raw_out; ok: the work row exists
template <int IN_KIND>
__device__ __forceinline__ void load_enc_row(RowInputs& in, const void* __restrict__ enc, int64_t r, bool ok)
{
	if (IN_KIND != NRF_MLP_IN_F32_CAT) {
		const uint4* e = reinterpret_cast<const uint4*>(enc) + r * 4;
#pragma unroll
		for (int q = 0; q < 4; q++) {
			const uint4 v = ok ? __ldg(e + q) : make_uint4(0u, 0u, 0u, 0u);
			in.e[4 * q] = v.x; in.e[4 * q + 1] = v.y; in.e[4 * q + 2] = v.z; in.e[4 * q + 3] = v.w;
		}
	} else {
		const float4* x = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(enc) + r * 48);
#pragma unroll
		for (int q = 0; q < 8; q++) {
			const float4 v = ok ? __ldg(x + q) : make_float4(0.f, 0.f, 0.f, 0.f);
			in.e[2 * q] = pack_f16(v.x, v.y);
			in.e[2 * q + 1] = pack_f16(v.z, v.w);
		}
	}
}

// w: the work row (ray = w / S); r: its position in enc / keep
template <int IN_KIND>
__device__ __forceinline__ void load_view_row(RowInputs& in, const void* __restrict__ enc, const float* __restrict__ ray_sh, int S,
	const uint8_t* __restrict__ keep, int64_t w, int64_t r, bool ok)
{
	in.kept = !(keep && ok && !keep[r]);
	if (IN_KIND == NRF_MLP_IN_ENC16_RAYBIAS) {   // the view term is a per-ray bias of the layer (add_ray_bias): K chunk 0 carries zeros
#pragma unroll
		for (int q = 0; q < 8; q++) in.v[q] = 0u;
		return;
	}
	const float4* vp = IN_KIND == NRF_MLP_IN_ENC16_RAYDIRS ? reinterpret_cast<const float4*>(ray_sh + (ok ? w / S : 0) * 16)
	                                                       : reinterpret_cast<const float4*>(reinterpret_cast<const float*>(enc) + (ok ? r : 0) * 48 + 32);
#pragma unroll
	for (int q = 0; q < 4; q++) {
		const float4 v = __ldg(vp + q);
		in.v[2 * q] = pack_f16(v.x, v.y);
		in.v[2 * q + 1] = pack_f16(v.z, v.w);
	}
}

// NRF_MLP_IN_ENC16_RAYBIAS: acc (32 fp32 accumulator bit patterns, columns c0 .. c0 + 31 of colour layer 0) += bias[ray][c0 ..]
__device__ __forceinline__ void add_ray_bias(uint32_t (&acc)[32], const float* __restrict__ bias_row, int c0)
{
	const float4* b = reinterpret_cast<const float4*>(bias_row + c0);
#pragma unroll
	for (int q = 0; q < 8; q++) {
		const float4 v = __ldg(b + q);
		acc[4 * q] = __float_as_uint(__uint_as_float(acc[4 * q]) + v.x);
		acc[4 * q + 1] = __float_as_uint(__uint_as_float(acc[4 * q + 1]) + v.y);
		acc[4 * q + 2] = __float_as_uint(__uint_as_float(acc[4 * q + 2]) + v.z);
		acc[4 * q + 3] = __float_as_uint(__uint_as_float(acc[4 * q + 3]) + v.w);
	}
}

template <int IN_KIND, bool MAPPED>
__global__ void __launch_bounds__(kThreads, 1) mlp_small_fwd_tc_kernel(const uint32_t* __restrict__ blob, const void* __restrict__ enc,
	const float* __restrict__ ray_sh, int S, const uint8_t* __restrict__ keep, int64_t n, RowMap map, float* __restrict__ raw_out)
{
	__shared__ Smem sm;
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int64_t n_tiles = (n + 127) / 128;

	if (warp == 0) {
		if (lane == 0) {
			mbar_init(&sm.w_ready, 1);
			for (int s = 0; s < kSlots; s++) { mbar_init(&sm.a_ready[s], 4); mbar_init(&sm.d_ready[s], 1); }
			asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
			// weights: one TMA bulk copy per CTA
			mbar_expect_tx(&sm.w_ready, kUmmaWords * 4);
			tma_bulk_g2s(sm.w, blob + kUmmaBase, kUmmaWords * 4, &sm.w_ready);
		}
		__syncwarp();
		tmem_alloc_all(&sm.tmem_base);
	}
	fence_before();
	__syncthreads();
	fence_after();
	const uint32_t tmem = sm.tmem_base;

	// ===== slot s = warps 4s..4s+3: one thread per row of the slot's 128-row tile; lane 0 of the slot's first warp also issues =====
	const int s = warp >> 2;
	const int row = ((warp & 3) << 5) | lane;                       // TMEM lane == row inside the tile
	const uint32_t col = tmem + s * kSlotCols;
	const uint32_t t_lane = col + (static_cast<uint32_t>((warp & 3) << 5) << 16);
	const bool issuer = (warp & 3) == 0 && lane == 0;
	uint64_t* const a_ready = &sm.a_ready[s];
	uint64_t* const d_ready = &sm.d_ready[s];
	const uint32_t w_saddr = smem_u32(sm.w);
	uint32_t pa = 0, pd = 0;                                        // phase parities of a_ready (issuer) / d_ready (everyone)
	const int64_t stride = static_cast<int64_t>(gridDim.x) * kSlots;
	int64_t tile = blockIdx.x + static_cast<int64_t>(gridDim.x) * s;

	RowInputs in;
	int64_t r_next = 0;                                             // position of the prefetched row in enc / keep / raw_out
	if (tile < n_tiles) {
		const int64_t w = tile * 128 + row;
		r_next = MAPPED ? merged_row(map, w, n) : w;
		load_enc_row<IN_KIND>(in, enc, r_next, w < n);
	}
	if (issuer) mbar_wait(&sm.w_ready, 0);

	for (; tile < n_tiles; tile += stride) {
		const int64_t w = tile * 128 + row;                         // work row
		const int64_t r = r_next;
		const bool ok = w < n;
		// ---- layer 0 operand
		tmem_st16(t_lane + kColA, in.e);
		publish(a_ready, lane);
		if (issuer) issue_layer<0>(a_ready, d_ready, pa, col, w_saddr);

		uint32_t acc0[32], acc1[32], a16[16];
		// ---- layer 0 -> h0 = relu(.) as the K=64 operand of layer 1
		mbar_wait(d_ready, pd); pd ^= 1u;
		fence_after();
		tmem_ld32(t_lane + kColD, acc0);
		tmem_ld32(t_lane + kColD + 32, acc1);
		tmem_ld_wait();
		relu_pack(acc0, a16);
		tmem_st16(t_lane + kColA, a16);
		relu_pack(acc1, a16);
		tmem_st16(t_lane + kColA + 16, a16);
		publish(a_ready, lane);
		if (issuer) issue_layer<1>(a_ready, d_ready, pa, col, w_saddr);
		// this row's view channels (per-ray SH table: cache hits) arrive while layer 1 runs
		load_view_row<IN_KIND>(in, enc, ray_sh, S, keep, w, r, ok);

		// ---- layer 1 -> [sigma | geo(15)]; colour input = [views(16) | 0 | geo(15)]
		mbar_wait(d_ready, pd); pd ^= 1u;
		fence_after();
		uint32_t d1[16];
		tmem_ld16(t_lane + kColD16, d1);
		tmem_ld_wait();
		const float sigma = __uint_as_float(d1[0]);
		d1[0] = 0u;                                                  // sigma slot of the colour input (its weight column is zero too)
#pragma unroll
		for (int i = 0; i < 8; i++) { a16[i] = in.v[i]; a16[8 + i] = pack_f16(__uint_as_float(d1[2 * i]), __uint_as_float(d1[2 * i + 1])); }
		tmem_st16(t_lane + kColA, a16);
		publish(a_ready, lane);
		const bool kept = in.kept;
		if (issuer) issue_layer<2>(a_ready, d_ready, pa, col, w_saddr);

		// ---- layers 2 and 3 -> relu -> K=64 operand of the next layer
#pragma unroll
		for (int l = 2; l <= 3; l++) {
			mbar_wait(d_ready, pd); pd ^= 1u;
			fence_after();
			tmem_ld32(t_lane + kColD, acc0);
			tmem_ld32(t_lane + kColD + 32, acc1);
			tmem_ld_wait();
			if (IN_KIND == NRF_MLP_IN_ENC16_RAYBIAS && l == 2) {
				const float* brow = ray_sh + (ok ? w / S : 0) * 64;
				add_ray_bias(acc0, brow, 0);
				add_ray_bias(acc1, brow, 32);
			}
			relu_pack(acc0, a16);
			tmem_st16(t_lane + kColA, a16);
			relu_pack(acc1, a16);
			tmem_st16(t_lane + kColA + 16, a16);
			publish(a_ready, lane);
			if (issuer) {
				if (l == 2) issue_layer<3>(a_ready, d_ready, pa, col, w_saddr);
				else issue_layer<4>(a_ready, d_ready, pa, col, w_saddr);
			}
			// next tile's encodings: in flight while this tile finishes its last two layers
			if (l == 2 && tile + stride < n_tiles) {
				const int64_t wn = (tile + stride) * 128 + row;
				r_next = MAPPED ? merged_row(map, wn, n) : wn;
				load_enc_row<IN_KIND>(in, enc, r_next, wn < n);
			}
		}

		// ---- layer 4 -> rgb; out = [r, g, b, sigma (0 outside the box, src/NeRFRenderer.h:188)]
		mbar_wait(d_ready, pd); pd ^= 1u;
		fence_after();
		uint32_t c[4];
		tmem_ld4(t_lane + kColD16, c);
		tmem_ld_wait();
		if (ok) *reinterpret_cast<float4*>(raw_out + r * 4) = make_float4(__uint_as_float(c[0]), __uint_as_float(c[1]), __uint_as_float(c[2]), kept ? sigma : 0.f);
	}

	fence_before();
	__syncthreads();
	if (warp == 0) {
		fence_after();
		tmem_free_all(tmem);
	}
}

}  // namespace tc

// called by nrf_mlp_small_fwd (mlp_small.cu)
cudaError_t launch_mlp_small_fwd_tc(const uint32_t* blob, int in_kind, const void* enc, const float* ray_sh, int S, const uint8_t* keep, int64_t n,
	float* raw_out, cudaStream_t stream)
{
	const int64_t tiles = (n + 127) / 128;
	const int blocks = static_cast<int>(std::min<int64_t>((tiles + tc::kSlots - 1) / tc::kSlots, kNumSMs));
	const tc::RowMap none{nullptr, 1, 1};
	if (in_kind == NRF_MLP_IN_ENC16_RAYDIRS)
		tc::mlp_small_fwd_tc_kernel<NRF_MLP_IN_ENC16_RAYDIRS, false><<<blocks, tc::kThreads, 0, stream>>>(blob, enc, ray_sh, S, keep, n, none, raw_out);
	else if (in_kind == NRF_MLP_IN_ENC16_RAYBIAS)
		tc::mlp_small_fwd_tc_kernel<NRF_MLP_IN_ENC16_RAYBIAS, false><<<blocks, tc::kThreads, 0, stream>>>(blob, enc, ray_sh, S, keep, n, none, raw_out);
	else
		tc::mlp_small_fwd_tc_kernel<NRF_MLP_IN_F32_CAT, false><<<blocks, tc::kThreads, 0, stream>>>(blob, enc, ray_sh, S, keep, n, none, raw_out);
	return cudaGetLastError();
}

// called by nrf_mlp_small_fwd_importance (mlp_small.cu): n = n_rays * n_importance work rows scattered over the merged arrays
cudaError_t launch_mlp_small_fwd_tc_importance(const uint32_t* blob, int in_kind, const void* enc, const float* ray_sh, const uint8_t* keep, const int16_t* perm,
	int64_t n_rays, int n_importance, int n_merged, float* raw_out, cudaStream_t stream)
{
	const int64_t n = n_rays * n_importance, tiles = (n + 127) / 128;
	const int blocks = static_cast<int>(std::min<int64_t>((tiles + tc::kSlots - 1) / tc::kSlots, kNumSMs));
	const tc::RowMap map{perm, n_importance, n_merged};
	if (in_kind == NRF_MLP_IN_ENC16_RAYBIAS)
		tc::mlp_small_fwd_tc_kernel<NRF_MLP_IN_ENC16_RAYBIAS, true><<<blocks, tc::kThreads, 0, stream>>>(blob, enc, ray_sh, n_importance, keep, n, map, raw_out);
	else
		tc::mlp_small_fwd_tc_kernel<NRF_MLP_IN_ENC16_RAYDIRS, true><<<blocks, tc::kThreads, 0, stream>>>(blob, enc, ray_sh, n_importance, keep, n, map, raw_out);
	return cudaGetLastError();
}

}  // namespace nrf
