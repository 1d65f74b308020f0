// Fused LeRF language head on tcgen05 / TMEM / TMA for sm_100a (SURVEY §8f-1, BASELINE C5).
//
// Replaces LeRFImpl::forward (reference src/LeRF.cpp:28-111: 4 bias-free cuBLAS SGEMMs + relu / index / cat / normalize kernels), the keep
// mask of LeRFRenderer::RunLENetwork (src/LeRFRenderer.cpp:18-20) and, with the two per-ray kernels at the end of this file, RenderCLIPEmbedding (src/LeRFRenderer.h:45-54) at
// the shape the reference trains (src/main.cpp:203-213 with the 512-d language dimension of C5): LeRF(geo 32, 2 layers, hidden 256, D 512) on
// the 16 x 8 = 128 channels of the language hash grid.
//
//   sigma net   h1 = relu(W_s0 enc)  [256]      s = W_s1 h1  [33] = [sigma_le | geo_feat 32]
//   language    h2 = relu(W_e0 [geo | enc])  [256]      e = W_e1 h2  [512]      out = [e / max(|e|, 1e-8) | sigma_le]
//
// Same mapping as mlp_nerf_tc.cu (one persistent CTA per SM, one 128-point tile in flight, A operands fp16 in TENSOR MEMORY, fp32 accumulators
// in TMEM, weights streamed through a 4 x 32 KB TMA ring as pre-packed UMMA K-major core matrices, warp 0 produces, warp 1 issues tcgen05.mma,
// warps 2..5 are one epilogue thread per row).  TMEM columns: D 0..255 | D2 (sigma head, N = 48) 256..303 | [geo 16 | enc 64] 304..383 (so the
// language net reads cat(geo, enc) as ONE contiguous K = 160 range, src/LeRF.cpp:96) | h 384..511.
//
// Three programs over the same kernel:
//   SIGMA   {S0, S1}: sigma_le only — the coarse pass of LeRFRenderer::RenderRays needs nothing else (its embedding is discarded,
//           src/LeRFRenderer.cpp:133-139).  Writes raw4 [N,4] = [0,0,0,sigma_le], the layout nrf_composite_fwd / nrf_sample_pdf_merge consume.
//   HIDDEN  {S0, S1, E0, G}: the fine pass.  The [N, 512] embedding is never formed: the rendered embedding is
//               normalize( sum_s w_s e_s / |e_s| ) = normalize( W_e1 * sum_s (w_s / |e_s|) h2_s )        (the last layer is linear),
//           and |e_s|^2 = h2_s^T G h2_s with G = W_e1^T W_e1 [256 x 256] built once by the pack kernel — a 256-wide layer instead of the
//           512-wide one.  Writes raw4, h2 (fp16 tile records, 512 B per row) and q = |e|^2 [N]; lerf_hsum_kernel + lerf_project_kernel finish per RAY.
//           (The reference materialises raw_le [R,S,513] fp32 = 2 KB per sample.)
//   RAW     {S0, S1, E0, E1 lower, E1 upper, E1 lower, E1 upper}: LeRF::forward itself, raw_le [N, 513] fp32.  The 512 outputs go through
//           the 256 accumulator columns in two halves, twice: the first pass only accumulates |e|^2, the second scales and stores
//           (through a per-warp shared-memory transpose, so a store instruction writes 128 contiguous bytes of one row).
// fp16 operands, fp32 accumulation: <= 1e-2 relative to the fp32 reference (tests/test_gpu_lerf.py).
#include "lerf_layout.cuh"
#include <algorithm>

namespace nrf {
namespace lerf_tc {

__constant__ ModeTable c_modes[kModes] = {make_mode(kSigma), make_mode(kHidden), make_mode(kRaw), make_mode(kTrain), make_mode(kChain)};
// padded logical weight Wp_l(n, k) in the kernel's operand order; gram = G = W_e1^T W_e1 (fp32 [256][256], lerf_gram_kernel)
__device__ __forceinline__ float wp(const Weights& p, const float* __restrict__ gram, int l, int n, int k, float g_inv)
{
	switch (l) {
		case 0: return p.s0[n * kIn + k];
		case 1: return n < kGeo ? p.s1[(n + 1) * kHid + k] : (n == kGeo ? p.s1[k] : 0.f);     // [geo 0..31 | sigma | zeros]
		case 2: return p.e0[n * (kGeo + kIn) + k];
		case 3: return gram[n * kHid + k] * g_inv;                                            // |G_nk| <= max diagonal <= 256 after scaling
		case 4: return p.e1[n * kHid + k];
		default: return p.e1[(n + 256) * kHid + k];
	}
}

// G[n][k] = sum_m W_e1[m][n] W_e1[m][k]: block = 4 rows n, thread = k; the four columns W_e1[.][n0..n0+3] are staged in shared memory, 16
// coalesced loads of W_e1[m][k] in flight per thread; fixed summation order (no atomics: the same weights must pack to the same bits).
// (The first pack kernel evaluated this 512-term sum once per packed word, twice: 108 us per optimiser step, profiles/r2_lerf_train_launches_v1.txt.)
__global__ void __launch_bounds__(kHid) lerf_gram_kernel(Weights p, float* __restrict__ gram)
{
	__shared__ __align__(16) float col[kDim][4];
	const int n0 = blockIdx.x * 4, k = threadIdx.x;
	for (int i = threadIdx.x; i < kDim * 4; i += kHid) col[i >> 2][i & 3] = p.e1[(i >> 2) * kHid + n0 + (i & 3)];
	__syncthreads();
	float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 16
	for (int m = 0; m < kDim; m++) {
		const float w = __ldg(p.e1 + m * kHid + k);
		const float4 c = *reinterpret_cast<const float4*>(&col[m][0]);
		acc[0] = fmaf(c.x, w, acc[0]); acc[1] = fmaf(c.y, w, acc[1]); acc[2] = fmaf(c.z, w, acc[2]); acc[3] = fmaf(c.w, w, acc[3]);
	}
#pragma unroll
	for (int i = 0; i < 4; i++) gram[(n0 + i) * kHid + k] = acc[i];
}

// scale of G: the smallest power of two s >= 1 with max_k G_kk / s <= 256 (|G_nk| <= sqrt(G_nn G_kk), so every entry fits fp16
// with 8 bits of headroom)
__global__ void __launch_bounds__(kHid) lerf_gscale_kernel(const float* __restrict__ gram, float* __restrict__ scale_out)
{
	__shared__ float red[kHid / 32];
	const int k = threadIdx.x;
	float d = gram[k * kHid + k];
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) d = fmaxf(d, __shfl_xor_sync(0xffffffffu, d, o));
	if ((k & 31) == 0) red[k >> 5] = d;
	__syncthreads();
	if (k == 0) {
		float mx = 0.f;
		for (int i = 0; i < kHid / 32; i++) mx = fmaxf(mx, red[i]);
		float sc = 1.f;
		while (mx > 256.f * sc && sc < 1e30f) sc *= 2.f;
		scale_out[0] = sc;
	}
}

__global__ void __launch_bounds__(256) lerf_pack_kernel(Weights p, uint32_t* __restrict__ blob)
{
	const int w = blockIdx.x * blockDim.x + threadIdx.x;
	if (w >= kScaleBase / 4) return;                       // the scale word is lerf_gscale_kernel's
	const float g_inv = 1.f / reinterpret_cast<const float*>(blob)[kScaleBase / 4];
	const float* const gram = reinterpret_cast<const float*>(blob) + kGramBase / 4;
	if (w >= kProjBase / 4) {
		const int i = w - kProjBase / 4, k = i / kDim, n = i % kDim;
		reinterpret_cast<float*>(blob)[w] = p.e1[n * kHid + k];
		return;
	}
	if (w >= kTrainBase / 4) {
		// the bf16 copy of S0, S1, E0, G: same stage layout as the fp16 copy below
		const int wt = w - kTrainBase / 4;
		int l = 0;
		while (l + 1 < 4 && wt * 4 >= layer_offset(l + 1)) l++;
		int q = wt - layer_offset(l) / 4, st = 0, k_off = 0;
		while (q >= stage_bytes(l, st) / 4) { q -= stage_bytes(l, st) / 4; k_off += stage_k(l, st); st++; }
		const auto [n, k] = stage_word(q, layer_info(l).N, k_off);
		// W_e0 travels with its input columns as [x 128 | geo 32] in the training copy (lerf_bwd_tc.cu: the two products that meet in d x then
		// write the same accumulator blocks); pairs (k, k + 1) never straddle the boundary
		const int ks = l == 2 ? (k < kIn ? k + kGeo : k - kIn) : k;
		blob[w] = pack_bf16(wp(p, gram, l, n, ks, g_inv), wp(p, gram, l, n, ks + 1, g_inv));
		return;
	}
	int l = 0;
	while (l + 1 < kLayers && w * 4 >= layer_offset(l + 1)) l++;
	int q = w - layer_offset(l) / 4, s = 0, k_off = 0;
	while (q >= stage_bytes(l, s) / 4) { q -= stage_bytes(l, s) / 4; k_off += stage_k(l, s); s++; }
	const auto [n, k] = stage_word(q, layer_info(l).N, k_off);
	blob[w] = pack_f16(wp(p, gram, l, n, k, g_inv), wp(p, gram, l, n, k + 1, g_inv));
}

struct __align__(128) Smem {
	uint8_t ring[kRing][kStageBytes];
	float tbuf[8][32][33];               // RAW: per-warp transpose of a 32 x 32 output block
	float xpart[2][128];                 // HV == 2: partial row sums exchanged between the two warps of a lane quarter
	uint64_t full[kRing], empty[kRing];
	uint64_t a_ready, d_ready;
	uint32_t tmem_base;
};

// Epilogue helpers.  HV = warps per TMEM lane quarter (1: four epilogue warps, one thread per row does all 256 accumulator columns;
// 2: eight warps, warps w and w + 4 share a quarter and each takes 128 columns).  c0 = first 32-column chunk of this warp, CH = 8 / HV chunks.

// relu(D) -> fp16 -> the h columns (the next layer's A operand); the tcgen05.ld of chunk c+1 is in flight while chunk c is converted and
// stored.  SAVE: the packed row also goes to the h2 tile record.
template <bool SAVE, int CH>
__device__ __forceinline__ void relu_to_h(uint32_t t_lane, uint8_t* __restrict__ rec_row, int c0)
{
	uint32_t acc0[32], acc1[32], a16[16];
	tmem_ld32(t_lane + kColD + 32 * c0, acc0);
#pragma unroll
	for (int cc = 0; cc < CH; cc += 2) {
		const int c = c0 + cc;
		tmem_ld_wait_for(acc0);
		tmem_ld32(t_lane + kColD + 32 * (c + 1), acc1);
#pragma unroll
		for (int i = 0; i < 16; i++) a16[i] = pack_f16_relu(__uint_as_float(acc0[2 * i]), __uint_as_float(acc0[2 * i + 1]));
		tmem_st16(t_lane + kColH + 16 * c, a16);
		if (SAVE) {
#pragma unroll
			for (int i = 0; i < 4; i++)
				*reinterpret_cast<uint4*>(rec_row + (4 * c + i) * 2048) = make_uint4(a16[4 * i], a16[4 * i + 1], a16[4 * i + 2], a16[4 * i + 3]);
		}
		tmem_ld_wait_for(acc1);
		if (cc + 2 < CH) tmem_ld32(t_lane + kColD + 32 * (c + 2), acc0);
#pragma unroll
		for (int i = 0; i < 16; i++) a16[i] = pack_f16_relu(__uint_as_float(acc1[2 * i]), __uint_as_float(acc1[2 * i + 1]));
		tmem_st16(t_lane + kColH + 16 * (c + 1), a16);
		if (SAVE) {
#pragma unroll
			for (int i = 0; i < 4; i++)
				*reinterpret_cast<uint4*>(rec_row + (4 * (c + 1) + i) * 2048) = make_uint4(a16[4 * i], a16[4 * i + 1], a16[4 * i + 2], a16[4 * i + 3]);
		}
	}
}

// sum of D^2 over this warp's accumulator columns (this thread's row)
template <int CH>
__device__ __forceinline__ float sumsq_d(uint32_t t_lane, int c0)
{
	uint32_t acc0[32], acc1[32];
	float s = 0.f;
	tmem_ld32(t_lane + kColD + 32 * c0, acc0);
#pragma unroll
	for (int cc = 0; cc < CH; cc += 2) {
		const int c = c0 + cc;
		tmem_ld_wait_for(acc0);
		tmem_ld32(t_lane + kColD + 32 * (c + 1), acc1);
#pragma unroll
		for (int i = 0; i < 32; i++) s = fmaf(__uint_as_float(acc0[i]), __uint_as_float(acc0[i]), s);
		tmem_ld_wait_for(acc1);
		if (cc + 2 < CH) tmem_ld32(t_lane + kColD + 32 * (c + 2), acc0);
#pragma unroll
		for (int i = 0; i < 32; i++) s = fmaf(__uint_as_float(acc1[i]), __uint_as_float(acc1[i]), s);
	}
	return s;
}

// TRAIN: relu(D) -> fp16 -> the h columns (the next layer's A operand); the row also goes to the bf16 record region (region_row = the row's first
// chunk of the region, chunks 1 KB apart: operand of the weight-gradient products) and, H16, to the fp16 region as well; BITS: the ReLU mask words
// of the row (8 x 32 bits, see lerf_layout.cuh)
template <bool BITS, bool H16>
__device__ __forceinline__ void relu_to_h_train(uint32_t t_lane, uint8_t* __restrict__ region_row, uint8_t* __restrict__ region16_row, uint32_t* __restrict__ bits_row)
{
	uint32_t acc0[32], acc1[32], a16[16], r16[16], words[8];
	tmem_ld32(t_lane + kColD, acc0);
#pragma unroll
	for (int c = 0; c < 8; c += 2) {
		tmem_ld_wait_for(acc0);
		tmem_ld32(t_lane + kColD + 32 * (c + 1), acc1);
#pragma unroll
		for (int half = 0; half < 2; half++) {
			uint32_t (&acc)[32] = half ? acc1 : acc0;
			if (half) {
				tmem_ld_wait_for(acc1);
				if (c + 2 < 8) tmem_ld32(t_lane + kColD + 32 * (c + 2), acc0);
			}
			uint32_t m = 0u;
#pragma unroll
			for (int i = 0; i < 16; i++) {
				a16[i] = pack_f16_relu(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1]));
				r16[i] = pack_bf16_relu(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1]));
				if (BITS) m |= ((a16[i] & 0xFFFFu) ? (1u << i) : 0u) | ((a16[i] >> 16) ? (1u << (16 + i)) : 0u);
			}
			words[c + half] = m;
			tmem_st16(t_lane + kColH + 16 * (c + half), a16);
#pragma unroll
			for (int i = 0; i < 4; i++) {
				*reinterpret_cast<uint4*>(region_row + (4 * (c + half) + i) * 1024) = make_uint4(r16[4 * i], r16[4 * i + 1], r16[4 * i + 2], r16[4 * i + 3]);
				if (H16) *reinterpret_cast<uint4*>(region16_row + (4 * (c + half) + i) * 1024) = make_uint4(a16[4 * i], a16[4 * i + 1], a16[4 * i + 2], a16[4 * i + 3]);
			}
		}
	}
	if (BITS) {
		reinterpret_cast<uint4*>(bits_row)[0] = make_uint4(words[0], words[1], words[2], words[3]);
		reinterpret_cast<uint4*>(bits_row)[1] = make_uint4(words[4], words[5], words[6], words[7]);
	}
}

// this warp's part of q = h^T (G h): D holds G h (fp32), the h columns hold h (fp16 pairs)
template <int CH, bool BF16 = false>
__device__ __forceinline__ float dot_d_h(uint32_t t_lane, int c0)
{
	uint32_t acc[32], hh[16];
	float s = 0.f;
#pragma unroll 1
	for (int c = c0; c < c0 + CH; c++) {
		tmem_ld32(t_lane + kColD + 32 * c, acc);
		tmem_ld16(t_lane + kColH + 16 * c, hh);
		tmem_ld_wait_for(acc);
		tmem_ld_wait_for(hh);
#pragma unroll
		for (int i = 0; i < 16; i++) {
			const float2 h2 = BF16 ? make_float2(__uint_as_float(hh[i] << 16), __uint_as_float(hh[i] & 0xFFFF0000u))
			                       : __half22float2(*reinterpret_cast<const __half2*>(&hh[i]));
			s = fmaf(h2.x, __uint_as_float(acc[2 * i]), s);
			s = fmaf(h2.y, __uint_as_float(acc[2 * i + 1]), s);
		}
	}
	return s;
}

// this warp's D columns * inv -> out[row, col0 + 32 c ..] (row stride 513 floats) through the warp's transpose buffer
template <int CH>
__device__ __forceinline__ void scaled_store(uint32_t t_lane, float inv, float (*tb)[33], int lane, int64_t warp_row0, int64_t n, float* __restrict__ out, int col0,
	int c0)
{
	uint32_t acc[32];
#pragma unroll 1
	for (int c = c0; c < c0 + CH; c++) {
		tmem_ld32(t_lane + kColD + 32 * c, acc);
		tmem_ld_wait_for(acc);
#pragma unroll
		for (int i = 0; i < 32; i++) tb[lane][i] = __uint_as_float(acc[i]) * inv;
		__syncwarp();
#pragma unroll 4
		for (int rr = 0; rr < 32; rr++) {
			const int64_t gr = warp_row0 + rr;
			if (gr < n) out[gr * (kDim + 1) + col0 + 32 * c + lane] = tb[rr][lane];
		}
		__syncwarp();
	}
}

// all epilogue threads (named barrier 1; warps 0 and 1 never take part)
template <int HV>
__device__ __forceinline__ void epilogue_sync()
{
	asm volatile("bar.sync 1, %0;" ::"n"(128 * HV) : "memory");
}

// epilogue warps per TMEM lane quarter: two for RAW (its 403 MB of 4-byte stores are instruction-bound: 331 -> 251 us), one otherwise
// (the TMEM read bandwidth, not the per-thread work, bounds those epilogues: 98.4 us with four warps, 102.0 us with eight)
__host__ __device__ constexpr int epi_warps_per_quarter(int mode) { return mode == kRaw ? 2 : 1; }

template <int MODE>
__global__ void __launch_bounds__(32 * (2 + 4 * epi_warps_per_quarter(MODE)), 1) lerf_fwd_tc_kernel(const uint8_t* __restrict__ blob, const uint4* __restrict__ enc,
	const uint8_t* __restrict__ keep, int64_t n, float* __restrict__ raw4, uint8_t* __restrict__ hidden, float* __restrict__ q_out, float* __restrict__ raw_le)
{
	extern __shared__ __align__(128) uint8_t smem_raw[];
	Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~uintptr_t(127));
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int64_t n_tiles = (n + 127) / 128;
	const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
	const ModeTable& mt = c_modes[MODE];
	constexpr int HV = epi_warps_per_quarter(MODE);
	constexpr int CH = 8 / HV;               // 32-column accumulator chunks per epilogue warp
	constexpr int PRE = 16 / HV;             // 16-byte pieces of the input row per epilogue thread
	constexpr uint32_t colEnc = kColEnc, colGeo = kColGeo;

	if (warp == 1) {
		if (lane == 0) {
			for (int s = 0; s < kRing; s++) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], 1); }
			mbar_init(&sm.a_ready, 4 * HV);
			mbar_init(&sm.d_ready, 1);
			asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		}
		__syncwarp();
		tmem_alloc_all(&sm.tmem_base);
	}
	fence_before();
	__syncthreads();
	fence_after();
	const uint32_t tmem = sm.tmem_base;

	if (warp == 0) {
		// ===== producer: the same weight-stage sequence for every tile =====
		if (lane == 0) {
			uint32_t g = 0;
			const int n_stages = mt.n_stages;
			for (int64_t t = 0; t < my_tiles; t++) {
#pragma unroll 1
				for (int i = 0; i < n_stages; i++, g++) {
					const uint32_t slot = g % kRing, round = g / kRing;
					mbar_wait(&sm.empty[slot], (round & 1u) ^ 1u);          // first round passes immediately
					const uint32_t bytes = mt.bytes[i];
					mbar_expect_tx(&sm.full[slot], bytes);
					tma_bulk_g2s(sm.ring[slot], blob + mt.off[i], bytes, &sm.full[slot]);
				}
			}
		}
	} else if (warp == 1) {
		// ===== MMA issuer =====
		if (lane == 0) {
			uint32_t g = 0, pa = 0;
			const int n_groups = mt.n_groups;
			for (int64_t t = 0; t < my_tiles; t++) {
#pragma unroll 1
				for (int grp = 0; grp < n_groups; grp++) {
					mbar_wait(&sm.a_ready, pa);
					pa ^= 1u;
					fence_after();
					const int l = mt.group_layer[grp];
					const LayerInfo L = layer_info(l);
					const uint32_t id = idesc(128, L.N, false, 0, 0);
					const uint32_t lbo = L.N * 16;
					uint32_t a_col = tmem + L.a_col;
					bool first = true;
					const int ns = layer_stages(l);
					for (int s = 0; s < ns; s++, g++) {
						const uint32_t slot = g % kRing, round = g / kRing;
						mbar_wait(&sm.full[slot], round & 1u);
						fence_after();
						const uint32_t saddr = smem_u32(sm.ring[slot]);
						const int ks = stage_k(l, s) / 16;
						for (int j = 0; j < ks; j++) {
							umma_ts(tmem + L.d_col, a_col, smem_desc(saddr + j * 2 * lbo, lbo, 128), id, first ? 0u : 1u);
							first = false;
							a_col += 8;
						}
						umma_commit(&sm.empty[slot]);                      // the stage is free again once these MMAs have read it
					}
					umma_commit(&sm.d_ready);
				}
			}
		}
	} else {
		// ===== epilogue warps: HV threads per row of the tile =====
		const int ew = warp - 2;
		const int qd = warp & 3;                                          // TMEM lane quarter this warp may access
		const int half = ew >> 2;                                         // which share of the columns (always 0 when HV == 1)
		const int c0 = half * CH;
		const int row = (qd << 5) | lane;
		const uint32_t t_lane = tmem + (static_cast<uint32_t>(qd << 5) << 16);
		uint32_t pd = 0;
		// The input row of the NEXT tile is requested while the last MMAs of the current tile run (PRE x 16 B per thread, held in registers):
		// at the top of a tile its global-load latency (the tensor pipe idle meanwhile) is already paid.
		uint4 pre[PRE];
		auto load_row = [&](int64_t tile_idx) {
			const int64_t rr = tile_idx * 128 + row;
			const bool in = tile_idx < n_tiles && rr < n;
			const uint4* er = enc + (in ? rr : 0) * (kIn / 8) + half * PRE;
#pragma unroll
			for (int i = 0; i < PRE; i++) pre[i] = in ? __ldg(er + i) : make_uint4(0u, 0u, 0u, 0u);
		};
		if (my_tiles > 0) load_row(blockIdx.x);
		for (int64_t t = 0; t < my_tiles; t++) {
			const int64_t tile = blockIdx.x + t * gridDim.x;
			const int64_t r = tile * 128 + row;
			const bool ok = r < n;
			// ---- input: the 128 fp16 channels of the language hash grid, as they leave nrf_hash_encode_fwd (already in registers, see load_row)
			// TRAIN: the HIDDEN program + every layer input also goes to the tile's record (hidden = the record base, lerf_layout.cuh)
			uint8_t* const rec = MODE == kTrain ? hidden + tile * static_cast<int64_t>(kSaveTile) : nullptr;
			{
				uint32_t a16[16];
#pragma unroll
				for (int h = 0; h < PRE / 4; h++) {
#pragma unroll
					for (int i = 0; i < 4; i++) {
						const uint4 v = pre[4 * h + i];
						a16[4 * i] = v.x; a16[4 * i + 1] = v.y; a16[4 * i + 2] = v.z; a16[4 * i + 3] = v.w;
					}
					if (MODE == kTrain) {
#pragma unroll
						for (int i = 0; i < 4; i++)      // x = columns 32..159 of the [geo | x] region (bf16 copy): chunks 4 + 4h + i
							*reinterpret_cast<uint4*>(rec + kSaveGX + chunk_offset(kGeo + kIn, row, 4 + 4 * h + i)) =
								make_uint4(half2_bits_to_bf16x2(a16[4 * i]), half2_bits_to_bf16x2(a16[4 * i + 1]), half2_bits_to_bf16x2(a16[4 * i + 2]),
									half2_bits_to_bf16x2(a16[4 * i + 3]));
					}
					tmem_st16(t_lane + colEnc + 4 * PRE * half + 16 * h, a16);
				}
			}
			publish(&sm.a_ready, lane);

			// ---- S0: h1 = relu(D)
			mbar_wait(&sm.d_ready, pd);
			pd ^= 1u;
			fence_after();
			if (MODE == kTrain) relu_to_h_train<true, false>(t_lane, rec + kSaveH1 + chunk_offset(kHid, row, 0), nullptr, reinterpret_cast<uint32_t*>(rec + kSaveBits1 + row * 32));
			else relu_to_h<false, CH>(t_lane, nullptr, c0);
			publish(&sm.a_ready, lane);
			if (MODE == kSigma) load_row(tile + gridDim.x);

			// ---- S1: [geo 32 | sigma] (48 columns: the first warp of each quarter)
			mbar_wait(&sm.d_ready, pd);
			pd ^= 1u;
			fence_after();
			float sigma = 0.f;
			if (half == 0) {
				uint32_t c4[4];
				tmem_ld4(t_lane + kColD2 + kGeo, c4);
				if (MODE != kSigma) {
					uint32_t acc[32], a16[16];
					tmem_ld32(t_lane + kColD2, acc);
					tmem_ld_wait_for(acc);
#pragma unroll
					for (int i = 0; i < 16; i++) a16[i] = pack_f16(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1]));
					tmem_st16(t_lane + colGeo, a16);
					if (MODE == kTrain) {
#pragma unroll
						for (int i = 0; i < 4; i++)      // geo = columns 0..31 of the [geo | x] region (bf16 copy)
							*reinterpret_cast<uint4*>(rec + kSaveGX + chunk_offset(kGeo + kIn, row, i)) =
								make_uint4(pack_bf16(__uint_as_float(acc[8 * i]), __uint_as_float(acc[8 * i + 1])), pack_bf16(__uint_as_float(acc[8 * i + 2]), __uint_as_float(acc[8 * i + 3])),
									pack_bf16(__uint_as_float(acc[8 * i + 4]), __uint_as_float(acc[8 * i + 5])), pack_bf16(__uint_as_float(acc[8 * i + 6]), __uint_as_float(acc[8 * i + 7])));
					}
				}
				tmem_ld_wait_for(c4);
				sigma = __uint_as_float(c4[0]);
				if (keep != nullptr && ok && keep[r] == 0) sigma = 0.f;               // src/LeRFRenderer.cpp:18-20
				if (MODE != kRaw) {
					if (ok) *reinterpret_cast<float4*>(raw4 + r * 4) = make_float4(0.f, 0.f, 0.f, sigma);
				}
			}
			if (MODE == kSigma) continue;       // the next tile's input stage is the next publish
			publish(&sm.a_ready, lane);

			// ---- E0: h2 = relu(D)
			mbar_wait(&sm.d_ready, pd);
			pd ^= 1u;
			fence_after();
			if (MODE == kHidden) relu_to_h<true, CH>(t_lane, hidden + tile * kHiddenTile + row * 16, c0);
			else if (MODE == kTrain) relu_to_h_train<false, true>(t_lane, rec + kSaveH2B + chunk_offset(kHid, row, 0), rec + kSaveH2 + chunk_offset(kHid, row, 0), nullptr);
			else relu_to_h<false, CH>(t_lane, nullptr, c0);
			publish(&sm.a_ready, lane);
			if (MODE == kHidden || MODE == kTrain) load_row(tile + gridDim.x);

			if (MODE == kHidden || MODE == kTrain) {
				// ---- G: |e|^2 = h2 . (G h2)
				mbar_wait(&sm.d_ready, pd);
				pd ^= 1u;
				fence_after();
				float qv = dot_d_h<CH>(t_lane, c0) * __ldg(reinterpret_cast<const float*>(blob + kScaleBase));     // G travels divided by this power of two
				if (HV > 1) {
					if (half != 0) sm.xpart[0][row] = qv;
					epilogue_sync<HV>();
					if (half == 0) qv += sm.xpart[0][row];
				}
				if (ok && half == 0) q_out[r] = qv;
			} else {
				// ---- E1, first pass: |e|^2 over both halves of the outputs
				float ss = 0.f;
#pragma unroll 1
				for (int pass = 0; pass < 2; pass++) {
					mbar_wait(&sm.d_ready, pd);
					pd ^= 1u;
					fence_after();
					ss += sumsq_d<CH>(t_lane, c0);
					publish(&sm.a_ready, lane);
				}
				if (HV > 1) {
					sm.xpart[half][row] = ss;
					epilogue_sync<HV>();
					ss = sm.xpart[0][row] + sm.xpart[1][row];
				}
				const float inv = 1.f / fmaxf(sqrtf(ss), 1e-8f);                      // F::normalize(eps 1e-8), src/LeRF.cpp:105
				load_row(tile + gridDim.x);
				// ---- E1, second pass: scale and store
#pragma unroll 1
				for (int pass = 0; pass < 2; pass++) {
					mbar_wait(&sm.d_ready, pd);
					pd ^= 1u;
					fence_after();
					scaled_store<CH>(t_lane, inv, sm.tbuf[ew], lane, tile * 128 + (qd << 5), n, raw_le, 256 * pass, c0);
					if (pass == 0) publish(&sm.a_ready, lane);
				}
				if (ok && half == 0) raw_le[r * (kDim + 1) + kDim] = sigma;           // src/LeRF.cpp:107-110
			}
		}
	}

	fence_before();
	__syncthreads();
	if (warp == 1) {
		fence_after();
		tmem_free_all(tmem);
	}
}

int check_shape(const nrf_lerf_shape* s)
{
	NRF_REQUIRE(s != nullptr, "shape is null");
	if (!(s->input_ch == kIn && s->hidden_dim == kHid && s->geo_feat_dim == kGeo && s->lang_embed_dim == kDim && s->num_layers == 2)) {
		set_error("nrf_lerf: only the BASELINE C5 shape LeRF(geo 32, 2 layers, hidden 256, D 512, in 128) is built");
		return NRF_ERR_UNSUPPORTED;
	}
	return NRF_OK;
}

template <int MODE>
static int launch(const nrf_lerf_shape* shape, const void* packed, const void* enc, const uint8_t* keep, int64_t n, float* raw4, void* hidden, float* q,
	float* raw_le, nrf_stream stream)
{
	if (int rc = check_shape(shape)) return rc;
	NRF_REQUIRE(n >= 0, "negative n");
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(packed && enc, "null pointer");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 127) == 0 && (reinterpret_cast<uintptr_t>(enc) & 15) == 0 && (reinterpret_cast<uintptr_t>(raw4) & 15) == 0 &&
		(reinterpret_cast<uintptr_t>(hidden) & 127) == 0, "packed / hidden must be 128-byte, enc / raw4 16-byte aligned");
	const int64_t tiles = (n + 127) / 128;
	const int smem = static_cast<int>(sizeof(Smem)) + 256;
	const int blocks = static_cast<int>(std::min<int64_t>(tiles, kNumSMs));
	constexpr int threads = 32 * (2 + 4 * epi_warps_per_quarter(MODE));
	NRF_CUDA(cudaFuncSetAttribute(lerf_fwd_tc_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
	lerf_fwd_tc_kernel<MODE><<<blocks, threads, smem, as_stream(stream)>>>(reinterpret_cast<const uint8_t*>(packed), reinterpret_cast<const uint4*>(enc), keep, n,
		raw4, reinterpret_cast<uint8_t*>(hidden), q, raw_le);
	NRF_CHECK_LAUNCH("lerf_fwd_tc_kernel");
	return NRF_OK;
}

// ---------------------------------------------------------------------------------------------------------------------------------------
// Per-ray finish of the HIDDEN program: Hs[ray] = sum_s (w_s / max(|e_s|, 1e-8)) h2_s, then rendered = normalize(W_e1 Hs, eps 1e-8)
// (src/LeRFRenderer.h:45-54 applied to the normalised embeddings of src/LeRF.cpp:105).

// one block per ray, 8 warps; warp v owns column chunks v, v+8, v+16, v+24 of the h2 records; lane = sample within a group of 32
// TRAIN: h2 comes from the training records (region layout, lerf_layout.cuh) instead of the inference records
template <bool TRAIN>
__global__ void __launch_bounds__(256) lerf_hsum_kernel(const float* __restrict__ weights, const uint4* __restrict__ hidden, const float* __restrict__ q,
	int32_t n_samples, float* __restrict__ hsum)
{
	extern __shared__ float cs[];
	const int64_t ray = blockIdx.x;
	for (int s = threadIdx.x; s < n_samples; s += blockDim.x) {
		const int64_t row = ray * n_samples + s;
		cs[s] = weights[row] / fmaxf(sqrtf(fmaxf(q[row], 0.f)), 1e-8f);
	}
	__syncthreads();
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (int j = warp; j < kHid / 8; j += 8) {
		float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
		for (int s = lane; s < n_samples; s += 32) {
			const int64_t row = ray * n_samples + s;
			const uint4 v = TRAIN ? __ldg(hidden + ((row >> 7) * static_cast<int64_t>(kSaveTile) + kSaveH2 + chunk_offset(kHid, static_cast<int>(row & 127), j)) / 16)
			                      : __ldg(hidden + (row >> 7) * (kHiddenTile / 16) + j * 128 + (row & 127));
			const float c = cs[s];
			const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
			for (int i = 0; i < 4; i++) {
				const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w4[i]));
				acc[2 * i] = fmaf(c, f.x, acc[2 * i]);
				acc[2 * i + 1] = fmaf(c, f.y, acc[2 * i + 1]);
			}
		}
#pragma unroll
		for (int i = 0; i < 8; i++) acc[i] = warp_sum(acc[i]);
		if (lane == 0) {
			float4* o = reinterpret_cast<float4*>(hsum + ray * kHid + j * 8);
			o[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
			o[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
		}
	}
}

// 4 rays per block, 256 threads: thread = (output quad oq = tid & 127, k half kh = tid >> 7) accumulates 4 rays x 4 outputs over its 128 k from
// W_e1^T (fp32 [256][512]: one 16-byte load per k, 512 contiguous bytes per warp, 8 in flight), the halves meet in shared memory, then each
// thread owns outputs tid and tid + 256 of every ray for the norm and the store.  (The first version — 8 rays per block, two scalar loads per k —
// was latency-bound on its 128 blocks: 60 us for 0.27 GFLOP.)
constexpr int kProjRays = 4;
__global__ void __launch_bounds__(256) lerf_project_kernel(const float* __restrict__ w_t, const float* __restrict__ hsum, int64_t n_rays, float* __restrict__ rendered,
	float* __restrict__ enorm)
{
	__shared__ float hs[kProjRays][kHid];
	__shared__ __align__(16) float red[2][kProjRays][kDim];
	__shared__ float part[8][kProjRays];
	const int64_t ray0 = static_cast<int64_t>(blockIdx.x) * kProjRays;
	for (int i = threadIdx.x; i < kProjRays * kHid; i += 256) {
		const int64_t ray = ray0 + i / kHid;
		hs[i / kHid][i % kHid] = ray < n_rays ? hsum[ray * kHid + i % kHid] : 0.f;
	}
	__syncthreads();
	const int oq = threadIdx.x & 127, kh = threadIdx.x >> 7;
	float4 acc[kProjRays];
#pragma unroll
	for (int i = 0; i < kProjRays; i++) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
	const float4* wq = reinterpret_cast<const float4*>(w_t) + oq;
#pragma unroll 8
	for (int k = kh * 128; k < kh * 128 + 128; k++) {
		const float4 w = __ldg(wq + k * (kDim / 4));
#pragma unroll
		for (int i = 0; i < kProjRays; i++) {
			const float h = hs[i][k];
			acc[i].x = fmaf(h, w.x, acc[i].x);
			acc[i].y = fmaf(h, w.y, acc[i].y);
			acc[i].z = fmaf(h, w.z, acc[i].z);
			acc[i].w = fmaf(h, w.w, acc[i].w);
		}
	}
#pragma unroll
	for (int i = 0; i < kProjRays; i++) *reinterpret_cast<float4*>(&red[kh][i][4 * oq]) = acc[i];
	__syncthreads();
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, j = threadIdx.x;
	float lo[kProjRays], hi[kProjRays];
#pragma unroll
	for (int i = 0; i < kProjRays; i++) {
		lo[i] = red[0][i][j] + red[1][i][j];
		hi[i] = red[0][i][256 + j] + red[1][i][256 + j];
		const float s = warp_sum(lo[i] * lo[i] + hi[i] * hi[i]);
		if (lane == 0) part[warp][i] = s;
	}
	__syncthreads();
#pragma unroll
	for (int i = 0; i < kProjRays; i++) {
		const int64_t ray = ray0 + i;
		if (ray >= n_rays) break;
		float ss = 0.f;
#pragma unroll
		for (int w = 0; w < 8; w++) ss += part[w][i];
		const float nrm = fmaxf(sqrtf(ss), 1e-8f);
		const float inv = 1.f / nrm;
		if (enorm != nullptr && j == 0) enorm[ray] = nrm;       // |W_e1 Hs|: the backward of the normalisation divides by it
		rendered[ray * kDim + j] = lo[i] * inv;
		rendered[ray * kDim + 256 + j] = hi[i] * inv;
	}
}

}  // namespace lerf_tc
}  // namespace nrf

using namespace nrf;
using namespace nrf::lerf_tc;

extern "C" {

int64_t nrf_lerf_packed_bytes(const nrf_lerf_shape* shape) { return lerf_tc::check_shape(shape) ? -1 : static_cast<int64_t>(kPackedBytes); }

int64_t nrf_lerf_hidden_bytes(const nrf_lerf_shape* shape, int64_t n)
{
	if (lerf_tc::check_shape(shape) || n < 0) return -1;
	return ((n + 127) / 128) * static_cast<int64_t>(kHiddenTile);
}

int nrf_lerf_pack(const nrf_lerf_shape* shape, const nrf_lerf_weights* w, void* packed, nrf_stream stream)
{
	if (int rc = lerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(w != nullptr && packed != nullptr, "null pointer");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 127) == 0, "packed blob must be 128-byte aligned");
	NRF_REQUIRE(w->sigma_w0 && w->sigma_w1 && w->le_w0 && w->le_w1, "null weight pointer");
	Weights p{w->sigma_w0, w->sigma_w1, w->le_w0, w->le_w1};
	float* const gram = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(packed) + kGramBase);
	lerf_gram_kernel<<<kHid / 4, kHid, 0, as_stream(stream)>>>(p, gram);
	NRF_CHECK_LAUNCH("lerf_gram_kernel");
	lerf_gscale_kernel<<<1, kHid, 0, as_stream(stream)>>>(gram, reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(packed) + kScaleBase));
	NRF_CHECK_LAUNCH("lerf_gscale_kernel");
	lerf_pack_kernel<<<(kScaleBase / 4 + 255) / 256, 256, 0, as_stream(stream)>>>(p, reinterpret_cast<uint32_t*>(packed));
	NRF_CHECK_LAUNCH("lerf_pack_kernel");
	return NRF_OK;
}

int nrf_lerf_fwd(const nrf_lerf_shape* shape, const void* packed, const void* enc_f16, const uint8_t* keep, int64_t n, float* raw_le, nrf_stream stream)
{
	if (int rc = lerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(n <= 0 || raw_le != nullptr, "null output");
	return launch<kRaw>(shape, packed, enc_f16, keep, n, nullptr, nullptr, nullptr, raw_le, stream);
}

int nrf_lerf_sigma_fwd(const nrf_lerf_shape* shape, const void* packed, const void* enc_f16, const uint8_t* keep, int64_t n, float* raw4, nrf_stream stream)
{
	if (int rc = lerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(n <= 0 || raw4 != nullptr, "null output");
	return launch<kSigma>(shape, packed, enc_f16, keep, n, raw4, nullptr, nullptr, nullptr, stream);
}

int nrf_lerf_hidden_fwd(const nrf_lerf_shape* shape, const void* packed, const void* enc_f16, const uint8_t* keep, int64_t n, float* raw4, void* hidden,
                        float* q, nrf_stream stream)
{
	if (int rc = lerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(n <= 0 || (raw4 && hidden && q), "null output");
	return launch<kHidden>(shape, packed, enc_f16, keep, n, raw4, hidden, q, nullptr, stream);
}

static int render_embedding_impl(bool train, const nrf_lerf_shape* shape, const void* packed, const float* weights, const void* hidden, const float* q, int64_t n_rays,
	int32_t n_samples, float* hsum, float* rendered, float* enorm, nrf_stream stream)
{
	if (int rc = lerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1 && n_samples <= 8192, "n_rays >= 0 and 1 <= n_samples <= 8192");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(packed && weights && hidden && q && hsum && rendered, "null pointer");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(hidden) & 15) == 0 && (reinterpret_cast<uintptr_t>(hsum) & 15) == 0, "hidden / hsum must be 16-byte aligned");
	if (train)
		lerf_hsum_kernel<true><<<static_cast<unsigned>(n_rays), 256, n_samples * sizeof(float), as_stream(stream)>>>(weights, reinterpret_cast<const uint4*>(hidden), q,
			n_samples, hsum);
	else
		lerf_hsum_kernel<false><<<static_cast<unsigned>(n_rays), 256, n_samples * sizeof(float), as_stream(stream)>>>(weights, reinterpret_cast<const uint4*>(hidden), q,
			n_samples, hsum);
	NRF_CHECK_LAUNCH("lerf_hsum_kernel");
	const float* w_t = reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(packed) + kProjBase);
	lerf_project_kernel<<<static_cast<unsigned>((n_rays + kProjRays - 1) / kProjRays), 256, 0, as_stream(stream)>>>(w_t, hsum, n_rays, rendered, enorm);
	NRF_CHECK_LAUNCH("lerf_project_kernel");
	return NRF_OK;
}

int nrf_lerf_render_embedding(const nrf_lerf_shape* shape, const void* packed, const float* weights, const void* hidden, const float* q, int64_t n_rays,
                              int32_t n_samples, float* hsum, float* rendered, nrf_stream stream)
{
	return render_embedding_impl(false, shape, packed, weights, hidden, q, n_rays, n_samples, hsum, rendered, nullptr, stream);
}

int64_t nrf_lerf_train_saved_bytes(const nrf_lerf_shape* shape, int64_t n)
{
	if (lerf_tc::check_shape(shape) || n < 0) return -1;
	return ((n + 127) / 128) * static_cast<int64_t>(kSaveTile);
}

int nrf_lerf_fwd_train(const nrf_lerf_shape* shape, const void* packed, const void* enc_f16, const uint8_t* keep, int64_t n, float* raw4, void* saved,
                       float* q, nrf_stream stream)
{
	if (int rc = lerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(n <= 0 || (raw4 && saved && q), "null output");
	return launch<kTrain>(shape, packed, enc_f16, keep, n, raw4, saved, q, nullptr, stream);
}

int nrf_lerf_render_embedding_train(const nrf_lerf_shape* shape, const void* packed, const float* weights, const void* saved, const float* q, int64_t n_rays,
                                    int32_t n_samples, float* hsum, float* rendered, float* enorm, nrf_stream stream)
{
	NRF_REQUIRE(n_rays <= 0 || enorm != nullptr, "null enorm");
	return render_embedding_impl(true, shape, packed, weights, saved, q, n_rays, n_samples, hsum, rendered, enorm, stream);
}

}
