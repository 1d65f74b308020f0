// Backward of the fused LeRF language head (SURVEY §8f-1, BASELINE C5) on tcgen05 / TMEM / TMA for sm_100a.
//
// Replaces what LibTorch autograd does behind LeRFImpl::forward (reference src/LeRF.cpp:78-110: 4 bias-free Linear layers + relu / cat /
// normalize), RenderCLIPEmbedding (src/LeRFRenderer.h:45-54) and the language loss (src/NeRFExecutor.h:957-983: huber(delta 1.25).sum(-1)
// .nanmean()): 8 cuBLAS SGEMMs over [N, 512]-wide activations + ~30 elementwise kernels.  Like the forward, the [N, 512] embedding is never
// formed.  With  a1 = W_s0 x, h1 = relu(a1), [sigma | g] = W_s1 h1, a2 = W_e0 [g | x], h2 = relu(a2), t = G h2 (G = W_e1^T W_e1), n = sqrt(h2.t),
// per ray  w = composite(sigma), c_s = w_s / n_s, Hs = sum_s c_s h2_s, E = W_e1 Hs, r = E / |E|  (oracle/restate.py:lerf_backward_fused_form,
// pinned against the reference's own modules under LibTorch autograd, tests/golden/lerf_grads.npz):
//
//   per ray   dE = (dr - r (r.dr)) / |E|,  u = W_e1^T dE [256],  dW_e1 += dE Hs^T                        lerf_ray_grad / lerf_u / lerf_outer kernels
//   per row   dw_s = (h2_s . u) / n_s  (-> nrf_composite_bwd gives d sigma),  beta_s = c_s dw_s / n_s         lerf_row_coef_kernel
//   chain     d h2 = c u - beta t,  d a2 = d h2 * [h2 > 0],  d[x | g] = d a2 W_e0,  d s = [d g | d sigma],     lerf_bwd_chain_kernel (tcgen05)
//             d h1 = d s W_s1,  d a1 = d h1 * [h1 > 0],  d x = d a1 W_s0 + d x(E0)  -> bf16 [N,128] for nrf_hash_encode_bwd (F = 8)
//   weights   dW_e0 = d a2^T [x | g],  dW_s1 = d s^T h1,  dW_s0 = d a1^T x,  P = sum_s beta_s h2_s h2_s^T      mlp_nerf_bwd_dw_kernel (tcgen05, dw_units.cuh)
//             dW_e1 -= W_e1 P                                                                               lerf_gram_apply_kernel
//
// The chain kernel is the mlp_nerf_bwd_chain_kernel design at 4 layers: one persistent CTA per SM, one 128-row tile in flight, warp 0 streams
// the bf16 FORWARD blob (its stage bytes read as an MN-major B operand give dY W without a transposed copy), warp 1 issues tcgen05.mma with the
// gradient rows as A operand in TMEM and fp32 accumulators in TMEM, warps 2..9 are two epilogue threads per row (half of the accumulator columns each).  TMEM columns:
//   D 0..255  (t = G h2 | then d[x 128 | g 32] in 0..159, onto which d a1 W_s0 is ACCUMULATED in 0..127)   | d s operand 160..183
//   A 256..383 (d a2, then d a1 written over the head of the d h1 accumulator once it has been read)  | h2 operand 384..511  | d h1 accumulator 256..511
// The bf16 blob packs W_e0 with its input columns as [x 128 | geo 32] so that the two products that meet in d x write the same 64-column
// accumulator blocks.  The forward and the G h2 product run on fp16 operands, gradient rows are bf16 (range), accumulation fp32; the weight-
// gradient products read bf16 copies of the activations (one tcgen05.mma cannot mix the formats).  Parity tests/test_gpu_lerf_train.py (rel 1e-2
// against fp64 at the kernels' rounding points).
#include "lerf_layout.cuh"
#include "dw_units.cuh"
#include <algorithm>

namespace nrf {
namespace lerf_tc {

__constant__ ModeTable c_chain = make_mode(kChain);

constexpr uint32_t kCD = 0, kCS = 160, kCA = 256, kCH2 = 384, kCD2 = 256;
constexpr int kChainThreads = 32 * 10;     // producer, issuer, 8 epilogue warps (two per TMEM lane quarter, half of the columns each)

struct __align__(128) ChainSmem {
	uint8_t ring[kRing][kStageBytes];
	uint64_t full[kRing], empty[kRing];
	uint64_t a_ready, d_ready;
	uint32_t tmem_base;
};

__global__ void __launch_bounds__(kChainThreads, 1) lerf_bwd_chain_kernel(const uint8_t* __restrict__ blob, const uint8_t* __restrict__ saved,
	const uint8_t* __restrict__ keep, const float* __restrict__ d_raw4, const float2* __restrict__ coef, const float* __restrict__ u, int32_t n_samples,
	int64_t n, uint8_t* __restrict__ grads, uint4* __restrict__ d_enc)
{
	extern __shared__ __align__(128) uint8_t smem_raw[];
	ChainSmem& sm = *reinterpret_cast<ChainSmem*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~uintptr_t(127));
	const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
	const int64_t n_tiles = (n + 127) / 128;
	const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

	if (warp == 1) {
		if (lane == 0) {
			for (int s = 0; s < kRing; s++) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], 1); }
			mbar_init(&sm.a_ready, 8);
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
		// ===== producer: G, E0, S1, S0 stages of the bf16 forward blob, every tile =====
		if (lane == 0) {
			uint32_t g = 0;
			const int n_stages = c_chain.n_stages;
			for (int64_t t = 0; t < my_tiles; t++) {
#pragma unroll 1
				for (int i = 0; i < n_stages; i++, g++) {
					const uint32_t slot = g % kRing, round = g / kRing;
					mbar_wait(&sm.empty[slot], (round & 1u) ^ 1u);
					const uint32_t bytes = c_chain.bytes[i];
					mbar_expect_tx(&sm.full[slot], bytes);
					tma_bulk_g2s(sm.ring[slot], blob + c_chain.off[i], bytes, &sm.full[slot]);
				}
			}
		}
	} else if (warp == 1) {
		// ===== MMA issuer: warp-uniform control flow, one elected lane issues =====
		const bool leader = elect_one();
		uint32_t g = 0, pa = 0;
		auto next_stage = [&]() -> uint32_t {
			const uint32_t slot = g % kRing, round = g / kRing;
			mbar_wait(&sm.full[slot], round & 1u);
			fence_after();
			g++;
			return slot;
		};
		for (int64_t t = 0; t < my_tiles; t++) {
			// ---- step 0: t = h2 G (fp16 operands, K-major B, as in the forward): 4 stages x 4 K steps, N = 256
			mbar_wait(&sm.a_ready, pa); pa ^= 1u; fence_after();
			{
				const uint32_t id = idesc(128, kHid, false, 0, 0), lbo = kHid * 16;
				uint32_t a_col = tmem + kCH2;
				for (int s = 0; s < 4; s++) {
					const uint32_t slot = next_stage();
					const uint32_t saddr = smem_u32(sm.ring[slot]);
					if (leader) {
#pragma unroll
						for (int j = 0; j < 4; j++) umma_ts(tmem + kCD, a_col + 8 * j, smem_desc(saddr + j * 2 * lbo, lbo, 128), id, (s | j) ? 1u : 0u);
						umma_commit(&sm.empty[slot]);
					}
					__syncwarp();
					a_col += 32;
				}
				if (leader) umma_commit(&sm.d_ready);
				__syncwarp();
			}
			// ---- step 1: d[x | g] = d a2 W_e0: stage s holds input columns 64 s .. of W_e0 -> accumulator block 64 s, complete over K = 256 outputs
			mbar_wait(&sm.a_ready, pa); pa ^= 1u; fence_after();
			for (int s = 0; s < 3; s++) {
				const uint32_t slot = next_stage();
				const uint64_t b0 = smem_desc(smem_u32(sm.ring[slot]), 128, kHid * 16);
				if (leader) {
					issue_k<16>(tmem + kCD + 64 * s, tmem + kCA, b0, idesc(128, s == 2 ? 32 : 64, true, 0, 1), 0u);
					umma_commit(&sm.empty[slot]);
				}
				__syncwarp();
			}
			if (leader) umma_commit(&sm.d_ready);
			__syncwarp();
			// ---- step 2: d h1 = d s W_s1: one stage (48 outputs x 256 inputs), K = 48, N = 256
			mbar_wait(&sm.a_ready, pa); pa ^= 1u; fence_after();
			{
				const uint32_t slot = next_stage();
				const uint64_t b0 = smem_desc(smem_u32(sm.ring[slot]), 128, kSigN * 16);
				if (leader) {
					issue_k<3>(tmem + kCD2, tmem + kCS, b0, idesc(128, kHid, true, 0, 1), 0u);
					umma_commit(&sm.empty[slot]);
					umma_commit(&sm.d_ready);
				}
				__syncwarp();
			}
			// ---- step 3: d x += d a1 W_s0: two stages of 64 input columns, accumulated onto the d x block of step 1
			mbar_wait(&sm.a_ready, pa); pa ^= 1u; fence_after();
			for (int s = 0; s < 2; s++) {
				const uint32_t slot = next_stage();
				const uint64_t b0 = smem_desc(smem_u32(sm.ring[slot]), 128, kHid * 16);
				if (leader) {
					issue_k<16>(tmem + kCD + 64 * s, tmem + kCA, b0, idesc(128, 64, true, 0, 1), 1u);
					umma_commit(&sm.empty[slot]);
				}
				__syncwarp();
			}
			if (leader) umma_commit(&sm.d_ready);
			__syncwarp();
		}
	} else {
		// ===== epilogue warps: two threads per row (warps w and w + 4 share a TMEM lane quarter; `half` takes column chunks 4 half .. 4 half + 3) =====
		const int qd = warp & 3, half = (warp - 2) >> 2;
		const int row = (qd << 5) | lane;
		const uint32_t t_lane = tmem + (static_cast<uint32_t>(qd << 5) << 16);
		const float gscale = __ldg(reinterpret_cast<const float*>(blob + kScaleBase));     // the G operand travels divided by this power of two
		uint32_t pd = 0;
		for (int64_t t = 0; t < my_tiles; t++) {
			const int64_t tile = blockIdx.x + t * gridDim.x;
			const int64_t r = tile * 128 + row;
			const bool ok = r < n;
			const uint8_t* const rec_s = saved + tile * static_cast<int64_t>(kSaveTile);
			uint8_t* const rec_g = grads + tile * static_cast<int64_t>(kGradTile);
			const float2 cb = ok ? __ldg(coef + r) : make_float2(0.f, 0.f);          // (c_s, beta_s)
			const float* const u_row = u + (ok ? r / n_samples : 0) * kHid;
			// ---- the h2 record row -> A operand of step 0
			{
				const uint8_t* h2_row = rec_s + kSaveH2 + chunk_offset(kHid, row, 0);
#pragma unroll
				for (int cc = 0; cc < 4; cc++) {
					const int c = 4 * half + cc;
					uint32_t a16[16];
#pragma unroll
					for (int i = 0; i < 4; i++) {
						const uint4 v = __ldg(reinterpret_cast<const uint4*>(h2_row + (4 * c + i) * 1024));
						a16[4 * i] = v.x; a16[4 * i + 1] = v.y; a16[4 * i + 2] = v.z; a16[4 * i + 3] = v.w;
					}
					tmem_st16(t_lane + kCH2 + 16 * c, a16);
				}
			}
			publish(&sm.a_ready, lane);

			// ---- step 0: d a2 = (c u - beta t) * [h2 > 0]  (-> A operand + record), beta h2 (-> record)
			mbar_wait(&sm.d_ready, pd); pd ^= 1u; fence_after();
			{
				uint8_t* const da2_row = rec_g + kGradA2 + chunk_offset(kHid, row, 0);
				uint8_t* const bh2_row = rec_g + kGradBH2 + chunk_offset(kHid, row, 0);
				const float bt = cb.y * gscale;
				uint32_t acc[2][32], hh[2][16];
				float4 uu[2][8];
				auto fetch = [&](int c, int b) {
					tmem_ld32(t_lane + kCD + 32 * c, acc[b]);
					tmem_ld16(t_lane + kCH2 + 16 * c, hh[b]);
#pragma unroll
					for (int i = 0; i < 8; i++) uu[b][i] = __ldg(reinterpret_cast<const float4*>(u_row + 32 * c) + i);
				};
				fetch(4 * half, 0);
#pragma unroll
				for (int cc = 0; cc < 4; cc++) {
					const int c = 4 * half + cc, b = cc & 1;
					tmem_ld_wait_for(acc[b]);
					tmem_ld_wait_for(hh[b]);
					if (cc + 1 < 4) fetch(c + 1, b ^ 1);         // the next chunk's TMEM / L1 reads fly under this chunk's arithmetic and stores
					uint32_t a16[16], b16[16];
#pragma unroll
					for (int i = 0; i < 16; i++) {
						const float u_lo = (i & 1) ? uu[b][i >> 1].z : uu[b][i >> 1].x, u_hi = (i & 1) ? uu[b][i >> 1].w : uu[b][i >> 1].y;
						const float2 hf = half2_bits_to_float2(hh[b][i]);        // h2 is stored / multiplied as fp16
						const float h_lo = hf.x, h_hi = hf.y;
						const float g_lo = h_lo > 0.f ? cb.x * u_lo - bt * __uint_as_float(acc[b][2 * i]) : 0.f;
						const float g_hi = h_hi > 0.f ? cb.x * u_hi - bt * __uint_as_float(acc[b][2 * i + 1]) : 0.f;
						a16[i] = pack_bf16(g_lo, g_hi);
						b16[i] = pack_bf16(cb.y * h_lo, cb.y * h_hi);
					}
					tmem_st16(t_lane + kCA + 16 * c, a16);
					store_chunks(da2_row, 4 * c, a16);
					store_chunks(bh2_row, 4 * c, b16);
				}
			}
			publish(&sm.a_ready, lane);

			// ---- step 1: d g (accumulator columns 128..159) -> d s = [d g 32 | d sigma | 0..] (48 columns: A operand of step 2 + record)
			mbar_wait(&sm.d_ready, pd); pd ^= 1u; fence_after();
			if (half == 0) {
				float d_sigma = ok ? __ldg(d_raw4 + r * 4 + 3) : 0.f;
				if (ok && keep != nullptr && keep[r] == 0) d_sigma = 0.f;             // sigma_le was overwritten with 0 there (src/LeRFRenderer.cpp:18-20)
				uint32_t acc[32], a16[16], tail[8];
				tmem_ld32(t_lane + kCD + 128, acc);
				tmem_ld_wait_for(acc);
#pragma unroll
				for (int i = 0; i < 16; i++) a16[i] = pack_bf16(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1]));
#pragma unroll
				for (int i = 0; i < 8; i++) tail[i] = 0u;
				tail[0] = pack_bf16(d_sigma, 0.f);
				tmem_st16(t_lane + kCS, a16);
				tmem_st8(t_lane + kCS + 16, tail);
				uint8_t* const ds_row = rec_g + kGradS + chunk_offset(kSigN, row, 0);
				store_chunks(ds_row, 0, a16);
				*reinterpret_cast<uint4*>(ds_row + 4 * 1024) = make_uint4(tail[0], 0u, 0u, 0u);
				*reinterpret_cast<uint4*>(ds_row + 5 * 1024) = make_uint4(0u, 0u, 0u, 0u);
			}
			publish(&sm.a_ready, lane);

			// ---- step 2: d a1 = d h1 * [h1 > 0] + record.  The bf16 pairs of chunk c go to columns 256 + 16 c: inside the accumulator columns of chunk
			// c / 2, which belong to the OTHER half for c >= 4 — so both halves first read all their chunks, meet, and only then overwrite.
			mbar_wait(&sm.d_ready, pd); pd ^= 1u; fence_after();
			{
				const uint4 bw = __ldg(reinterpret_cast<const uint4*>(rec_s + kSaveBits1 + row * 32) + half);
				const uint32_t bits[4] = {bw.x, bw.y, bw.z, bw.w};
				uint8_t* const da1_row = rec_g + kGradA1 + chunk_offset(kHid, row, 0);
				uint32_t packed[4][16];
				uint32_t acc[2][32];
				tmem_ld32(t_lane + kCD2 + 32 * (4 * half), acc[0]);
#pragma unroll
				for (int cc = 0; cc < 4; cc++) {
					const int c = 4 * half + cc, b = cc & 1;
					tmem_ld_wait_for(acc[b]);
					if (cc + 1 < 4) tmem_ld32(t_lane + kCD2 + 32 * (c + 1), acc[b ^ 1]);
#pragma unroll
					for (int i = 0; i < 16; i++) {
						uint32_t w = pack_bf16(__uint_as_float(acc[b][2 * i]), __uint_as_float(acc[b][2 * i + 1]));
						w &= ((bits[cc] >> i) & 0x00010001u) * 0xFFFFu;
						packed[cc][i] = w;
					}
					store_chunks(da1_row, 4 * c, packed[cc]);
				}
				fence_before();
				asm volatile("bar.sync 1, 256;" ::: "memory");       // all 8 epilogue warps: every tcgen05.ld of the d h1 accumulator has completed
				fence_after();
#pragma unroll
				for (int cc = 0; cc < 4; cc++) tmem_st16(t_lane + kCA + 16 * (4 * half + cc), packed[cc]);
			}
			publish(&sm.a_ready, lane);

			// ---- step 3: d x (accumulator columns 0..127) -> bf16 [N, 128] row-major, the layout nrf_hash_encode_bwd reads
			mbar_wait(&sm.d_ready, pd); pd ^= 1u; fence_after();
			{
				uint32_t acc[2][32];
				tmem_ld32(t_lane + kCD + 32 * (2 * half), acc[0]);
				tmem_ld32(t_lane + kCD + 32 * (2 * half + 1), acc[1]);
#pragma unroll
				for (int cc = 0; cc < 2; cc++) {
					const int c = 2 * half + cc;
					uint32_t a16[16];
					tmem_ld_wait_for(acc[cc]);
#pragma unroll
					for (int i = 0; i < 16; i++) a16[i] = pack_bf16(__uint_as_float(acc[cc][2 * i]), __uint_as_float(acc[cc][2 * i + 1]));
					if (ok) {
#pragma unroll
						for (int i = 0; i < 4; i++) d_enc[r * (kIn / 8) + 4 * c + i] = make_uint4(a16[4 * i], a16[4 * i + 1], a16[4 * i + 2], a16[4 * i + 3]);
					}
				}
				// every tcgen05.ld of this tile has completed: the next tile's h2 operand may overwrite columns 384.. (and step 0's MMAs column 0..)
				fence_before();
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

// ---- per-ray kernels ---------------------------------------------------------------------------------------------------------------------

// One block per ray.  d r: either given (grad_rendered, any loss) or formed here from the reference's language loss (target; huber delta 1.25
// summed over the 512 channels, mean over the rays, src/NeRFExecutor.h:964-968; loss_out += this ray's share).  Then the backward of
// r = E / max(|E|, 1e-8):  dE = (dr - r (r . dr)) / |E|.
__global__ void __launch_bounds__(256) lerf_ray_grad_kernel(const float* __restrict__ rendered, const float* __restrict__ enorm, const float* __restrict__ target,
	const float* __restrict__ grad_rendered, float inv_rays, float grad_scale, float* __restrict__ loss_out, float* __restrict__ d_e)
{
	__shared__ float red[2][8];
	const int64_t ray = blockIdx.x;
	const int j = threadIdx.x;
	float rr[2], dr[2], loss = 0.f, dot = 0.f;
#pragma unroll
	for (int h = 0; h < 2; h++) {
		const int64_t idx = ray * kDim + j + 256 * h;
		rr[h] = rendered[idx];
		if (grad_rendered != nullptr) {
			dr[h] = grad_rendered[idx] * grad_scale;
		} else {
			const float e = rr[h] - target[idx];
			const float ae = fabsf(e);
			loss += ae < 1.25f ? 0.5f * e * e : 1.25f * (ae - 0.625f);
			dr[h] = (ae < 1.25f ? e : (e > 0.f ? 1.25f : -1.25f)) * inv_rays * grad_scale;
		}
		dot = fmaf(rr[h], dr[h], dot);
	}
	loss = warp_sum(loss);
	dot = warp_sum(dot);
	if ((j & 31) == 0) { red[0][j >> 5] = loss; red[1][j >> 5] = dot; }
	__syncthreads();
	float l = 0.f, d = 0.f;
#pragma unroll
	for (int w = 0; w < 8; w++) { l += red[0][w]; d += red[1][w]; }
	if (j == 0 && loss_out != nullptr && grad_rendered == nullptr) atomicAdd(loss_out, l * inv_rays);
	const float nrm = enorm[ray];
	const bool clamped = !(nrm > 1e-8f);                           // F::normalize's eps branch: r = E / eps, no projection
#pragma unroll
	for (int h = 0; h < 2; h++) d_e[ray * kDim + j + 256 * h] = (clamped ? dr[h] : dr[h] - rr[h] * d) / nrm;
}

// u[ray, k] = sum_n dE[ray, n] W_e1[n, k]: 8 rays per block, thread = k.  dE sits transposed in shared memory ([n][ray]: a thread reads its 8
// rays' values as two 16-byte broadcasts) and 16 weight loads are in flight per thread.  No atomics: u feeds d_enc, whose bits must not depend on
// scheduling (chunked / whole-batch equality, tests/test_gpu_lerf_train.py).  (First version: [ray][n] tile, 8 scalar LDS per n: 73 us.)
constexpr int kURays = 8;
__global__ void __launch_bounds__(256) lerf_u_kernel(const float* __restrict__ w_e1, const float* __restrict__ d_e, int64_t n_rays, float* __restrict__ u)
{
	__shared__ __align__(16) float de[kDim][kURays];
	const int64_t ray0 = static_cast<int64_t>(blockIdx.x) * kURays;
	for (int i = threadIdx.x; i < kURays * kDim; i += 256) {
		const int rr = i / kDim, nn = i % kDim;
		de[nn][rr] = ray0 + rr < n_rays ? d_e[(ray0 + rr) * kDim + nn] : 0.f;
	}
	__syncthreads();
	float acc[kURays];
#pragma unroll
	for (int i = 0; i < kURays; i++) acc[i] = 0.f;
	const int k = threadIdx.x;
#pragma unroll 16
	for (int nn = 0; nn < kDim; nn++) {
		const float w = __ldg(w_e1 + nn * kHid + k);
		const float4 a = *reinterpret_cast<const float4*>(&de[nn][0]), b = *reinterpret_cast<const float4*>(&de[nn][4]);
		acc[0] = fmaf(a.x, w, acc[0]); acc[1] = fmaf(a.y, w, acc[1]); acc[2] = fmaf(a.z, w, acc[2]); acc[3] = fmaf(a.w, w, acc[3]);
		acc[4] = fmaf(b.x, w, acc[4]); acc[5] = fmaf(b.y, w, acc[5]); acc[6] = fmaf(b.z, w, acc[6]); acc[7] = fmaf(b.w, w, acc[7]);
	}
#pragma unroll
	for (int i = 0; i < kURays; i++)
		if (ray0 + i < n_rays) u[(ray0 + i) * kHid + k] = acc[i];
}

// dW_e1[n, k] += sum_ray dE[ray, n] Hs[ray, k]: block = (8 output rows, a slice of the rays), thread = k
constexpr int kOuterRows = 8, kOuterSplit = 8;
__global__ void __launch_bounds__(256) lerf_outer_kernel(const float* __restrict__ d_e, const float* __restrict__ hsum, int64_t n_rays, float* __restrict__ g_e1)
{
	const int n0 = blockIdx.x * kOuterRows, k = threadIdx.x;
	const int64_t per = (n_rays + kOuterSplit - 1) / kOuterSplit;
	const int64_t lo = blockIdx.y * per, hi = lo + per < n_rays ? lo + per : n_rays;
	float acc[kOuterRows];
#pragma unroll
	for (int i = 0; i < kOuterRows; i++) acc[i] = 0.f;
#pragma unroll 4
	for (int64_t ray = lo; ray < hi; ray++) {
		const float hs = __ldg(hsum + ray * kHid + k);
		const float4 a = __ldg(reinterpret_cast<const float4*>(d_e + ray * kDim + n0)), b = __ldg(reinterpret_cast<const float4*>(d_e + ray * kDim + n0) + 1);
		acc[0] = fmaf(a.x, hs, acc[0]); acc[1] = fmaf(a.y, hs, acc[1]); acc[2] = fmaf(a.z, hs, acc[2]); acc[3] = fmaf(a.w, hs, acc[3]);
		acc[4] = fmaf(b.x, hs, acc[4]); acc[5] = fmaf(b.y, hs, acc[5]); acc[6] = fmaf(b.z, hs, acc[6]); acc[7] = fmaf(b.w, hs, acc[7]);
	}
#pragma unroll
	for (int i = 0; i < kOuterRows; i++) atomicAdd(g_e1 + (n0 + i) * kHid + k, acc[i]);
}

// One block per ray: dw_s = (h2_s . u_ray) / n_s,  c_s = w_s / n_s,  beta_s = c_s dw_s / n_s  (n_s = max(sqrt(q_s), 1e-8)).
// Warp v owns column chunks v, v + 8, v + 16, v + 24 of the h2 records (lerf_hsum_kernel's access pattern); lane = sample within a group of 32.
__global__ void __launch_bounds__(256) lerf_row_coef_kernel(const float* __restrict__ weights, const uint4* __restrict__ saved, const float* __restrict__ q,
	const float* __restrict__ u, int32_t n_samples, float* __restrict__ dw, float2* __restrict__ coef)
{
	extern __shared__ float sh[];                 // [256] u_ray, then [8][n_samples] partial dots
	float* const us = sh;
	float* const part = sh + kHid;
	const int64_t ray = blockIdx.x;
	us[threadIdx.x] = u[ray * kHid + threadIdx.x];
	__syncthreads();
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for (int s = lane; s < n_samples; s += 32) {
		const int64_t row = ray * n_samples + s;
		float acc = 0.f;
#pragma unroll
		for (int jj = 0; jj < 4; jj++) {
			const int j = warp + 8 * jj;
			const uint4 v = __ldg(saved + ((row >> 7) * static_cast<int64_t>(kSaveTile) + kSaveH2 + chunk_offset(kHid, static_cast<int>(row & 127), j)) / 16);
			const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
			for (int i = 0; i < 4; i++) {
				const float2 hf = half2_bits_to_float2(w4[i]);
				acc = fmaf(hf.x, us[8 * j + 2 * i], acc);
				acc = fmaf(hf.y, us[8 * j + 2 * i + 1], acc);
			}
		}
		part[warp * n_samples + s] = acc;
	}
	__syncthreads();
	for (int s = threadIdx.x; s < n_samples; s += blockDim.x) {
		float dot = 0.f;
#pragma unroll
		for (int w = 0; w < 8; w++) dot += part[w * n_samples + s];
		const int64_t row = ray * n_samples + s;
		const float nrm = fmaxf(sqrtf(fmaxf(q[row], 0.f)), 1e-8f);
		const float c = weights[row] / nrm, d = dot / nrm;
		dw[row] = d;
		coef[row] = make_float2(c, c * d / nrm);
	}
}

// dW_e1[i, n] -= sum_m W_e1[i, m] P[m, n]: block = output row i, thread = n
__global__ void __launch_bounds__(256) lerf_gram_apply_kernel(const float* __restrict__ w_e1, const float* __restrict__ gram, float* __restrict__ g_e1)
{
	__shared__ float wrow[kHid];
	const int i = blockIdx.x, nn = threadIdx.x;
	wrow[nn] = w_e1[i * kHid + nn];
	__syncthreads();
	float acc = 0.f;
#pragma unroll 8
	for (int m = 0; m < kHid; m++) acc = fmaf(wrow[m], __ldg(gram + m * kHid + nn), acc);
	g_e1[i * kHid + nn] -= acc;
}

// workspace: [gradient records | dE [R,512] | u [R,256] | coef [N] float2 | P [256,256]]
struct Workspace {
	uint8_t* grads;
	float* d_e;
	float* u;
	float2* coef;
	float* gram;
};
static int64_t align256(int64_t v) { return (v + 255) & ~int64_t(255); }
static int64_t carve(void* base, int64_t n, int64_t n_rays, Workspace* w)
{
	uint8_t* p = reinterpret_cast<uint8_t*>(base);
	int64_t off = 0;
	auto take = [&](int64_t bytes) { uint8_t* r = p ? p + off : nullptr; off += align256(bytes); return r; };
	uint8_t* g = take(((n + 127) / 128) * static_cast<int64_t>(kGradTile));
	uint8_t* de = take(n_rays * kDim * 4);
	uint8_t* uu = take(n_rays * kHid * 4);
	uint8_t* cf = take(n * 8);
	uint8_t* gr = take(kHid * kHid * 4);
	if (w) { w->grads = g; w->d_e = reinterpret_cast<float*>(de); w->u = reinterpret_cast<float*>(uu); w->coef = reinterpret_cast<float2*>(cf); w->gram = reinterpret_cast<float*>(gr); }
	return off;
}

}  // namespace lerf_tc
}  // namespace nrf

using namespace nrf;
using namespace nrf::lerf_tc;

extern "C" {

int64_t nrf_lerf_bwd_workspace_bytes(const nrf_lerf_shape* shape, int64_t n, int64_t n_rays)
{
	if (lerf_tc::check_shape(shape) || n < 0 || n_rays < 0) return -1;
	return carve(nullptr, n, n_rays, nullptr);
}

int nrf_lerf_bwd_rays(const nrf_lerf_shape* shape, const nrf_lerf_weights* weights, const void* saved, const float* q, const float* comp_weights,
	const float* hsum, const float* rendered, const float* enorm, const float* target, const float* grad_rendered, int64_t n_rays, int32_t n_samples,
	float grad_scale, float* loss_out, float* grad_le_w1, void* workspace, float* dw_out, nrf_stream stream)
{
	if (int rc = lerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1 && n_samples <= 8192, "n_rays >= 0 and 1 <= n_samples <= 8192");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(weights && weights->le_w1 && saved && q && comp_weights && hsum && rendered && enorm && workspace && dw_out && grad_le_w1, "null pointer");
	NRF_REQUIRE((target != nullptr) != (grad_rendered != nullptr), "exactly one of target / grad_rendered");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(saved) & 127) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "saved must be 128-byte, workspace 256-byte aligned");
	Workspace w;
	carve(workspace, n_rays * n_samples, n_rays, &w);
	cudaStream_t s = as_stream(stream);
	lerf_ray_grad_kernel<<<static_cast<unsigned>(n_rays), 256, 0, s>>>(rendered, enorm, target, grad_rendered, 1.f / static_cast<float>(n_rays), grad_scale, loss_out, w.d_e);
	NRF_CHECK_LAUNCH("lerf_ray_grad_kernel");
	lerf_u_kernel<<<static_cast<unsigned>((n_rays + kURays - 1) / kURays), 256, 0, s>>>(weights->le_w1, w.d_e, n_rays, w.u);
	NRF_CHECK_LAUNCH("lerf_u_kernel");
	lerf_outer_kernel<<<dim3(kDim / kOuterRows, kOuterSplit), 256, 0, s>>>(w.d_e, hsum, n_rays, grad_le_w1);
	NRF_CHECK_LAUNCH("lerf_outer_kernel");
	const size_t smem = (kHid + 8 * n_samples) * sizeof(float);
	if (smem > 48 * 1024) NRF_CUDA(cudaFuncSetAttribute(lerf_row_coef_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
	lerf_row_coef_kernel<<<static_cast<unsigned>(n_rays), 256, smem, s>>>(comp_weights, reinterpret_cast<const uint4*>(saved), q, w.u, n_samples, dw_out, w.coef);
	NRF_CHECK_LAUNCH("lerf_row_coef_kernel");
	return NRF_OK;
}

int nrf_lerf_bwd_rows(const nrf_lerf_shape* shape, const void* packed, const nrf_lerf_weights* weights, const void* saved, const uint8_t* keep,
	const float* d_raw4, int64_t n, int32_t n_samples, void* workspace, const nrf_lerf_weights* grads, void* d_enc_bf16, nrf_stream stream)
{
	if (int rc = lerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(n >= 0 && n_samples >= 1 && n % n_samples == 0, "n must be n_rays * n_samples");
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(packed && weights && weights->le_w1 && saved && d_raw4 && workspace && grads && d_enc_bf16, "null pointer");
	NRF_REQUIRE(grads->sigma_w0 && grads->sigma_w1 && grads->le_w0 && grads->le_w1, "null gradient pointer");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 127) == 0 && (reinterpret_cast<uintptr_t>(saved) & 127) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0 &&
		(reinterpret_cast<uintptr_t>(d_enc_bf16) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_raw4) & 15) == 0, "packed / saved must be 128-byte, workspace 256-byte, d_enc / d_raw4 16-byte aligned");
	Workspace w;
	carve(workspace, n, n / n_samples, &w);
	cudaStream_t s = as_stream(stream);
	const int64_t tiles = (n + 127) / 128;
	{
		const int blocks = static_cast<int>(std::min<int64_t>(tiles, kNumSMs));
		const int smem = static_cast<int>(sizeof(ChainSmem)) + 256;
		NRF_CUDA(cudaFuncSetAttribute(lerf_bwd_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
		lerf_bwd_chain_kernel<<<blocks, kChainThreads, smem, s>>>(reinterpret_cast<const uint8_t*>(packed), reinterpret_cast<const uint8_t*>(saved), keep, d_raw4,
			w.coef, w.u, n_samples, n, w.grads, reinterpret_cast<uint4*>(d_enc_bf16));
		NRF_CHECK_LAUNCH("lerf_bwd_chain_kernel");
	}
	NRF_CUDA(cudaMemsetAsync(w.gram, 0, kHid * kHid * sizeof(float), s));
	{
		float* const ge0 = const_cast<float*>(grads->le_w0);
		float* const gs0 = const_cast<float*>(grads->sigma_w0);
		float* const gs1 = const_cast<float*>(grads->sigma_w1);
		dw::UnitTable T{};
		int c = 0;
		auto unit = [&](int a_src, int a_off, int a_cols, int b_src, int b_off, int b_cols, int b_half, int n_lo, int n_hi, int stride_m, int stride_n, float* out) -> dw::Unit& {
			dw::Unit& U = T.u[c++];
			U.a_src = a_src; U.a_off = a_off; U.a_cols = a_cols;
			U.b_src = b_src; U.b_off = b_off; U.b_cols = b_cols; U.b_half = b_half;
			U.n_lo = n_lo; U.n_hi = n_hi; U.stride_m = stride_m; U.stride_n = stride_n; U.out = out;
			return U;
		};
		// all operands bf16: the gradient rows written by the chain, and the bf16 copies of the activations saved by the forward
		// dW_e0 [256, 160] = d a2^T [geo 32 | x 128]
		unit(0, kGradA2, kHid, 1, kSaveGX, kGeo + kIn, 0, 0, kGeo + kIn, kGeo + kIn, 1, ge0);
		// dW_s0 [256, 128] = d a1^T x: x = columns 32..159 of the [geo | x] region
		unit(0, kGradA1, kHid, 1, kSaveGX + (kGeo / 8) * 1024, kIn, (kGeo + kIn) * 128, 0, kIn, kIn, 1, gs0);
		// dW_s1 [33, 256], roles swapped (M = input index): D[m, n] = sum h1[., m] d s[., n]; n < 32 -> row n + 1 (geo), n = 32 -> row 0 (sigma)
		{
			dw::Unit& U = unit(1, kSaveH1, kHid, 0, kGradS, kSigN, 0, 0, kGeo, 1, kHid, gs1 + kHid);
			U.n2_lo = kGeo; U.n2_hi = kGeo + 1; U.out2 = gs1;
		}
		// P [256, 256] = (beta h2)^T h2
		unit(0, kGradBH2, kHid, 1, kSaveH2B, kHid, 0, 0, kHid, kHid, 1, w.gram);
		T.count = c;
		T.save_tile = kSaveTile;
		T.grad_tile = kGradTile;
		if (int rc = dw::launch_dw_units(T, saved, w.grads, tiles, stream)) return rc;
	}
	lerf_gram_apply_kernel<<<kDim, kHid, 0, s>>>(weights->le_w1, w.gram, const_cast<float*>(grads->le_w1));
	NRF_CHECK_LAUNCH("lerf_gram_apply_kernel");
	return NRF_OK;
}

}
