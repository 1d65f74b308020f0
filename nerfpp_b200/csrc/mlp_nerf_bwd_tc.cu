// Backward of the classic NeRF MLP (NeRFImpl::forward, reference src/NeRF.cpp:92-126, differentiated by LibTorch autograd in the
// reference: 11 cuBLAS SGEMM pairs + ReLU-mask / bias-sum kernels, SURVEY §8a-a7) on tcgen05 / TMEM / TMA for sm_100a.
//
// Two kernels over the scratch records of mlp_nerf_layout.cuh (written by nrf_mlp_nerf_fwd_train):
//
//  1. mlp_nerf_bwd_chain_kernel — the gradient chain  dY_{l-1} = (dY_l W_l) * relu'(h_l), one persistent CTA per SM, one 128-row tile
//     in flight.  Same roles as the forward: warp 0 streams the FORWARD weight blob through a 4 x 32 KB TMA ring (38 of its 41
//     stages, in reverse layer order; the stage bytes are read as an MN-major B operand, so no transposed copy of the weights
//     exists), warp 1 issues tcgen05.mma M=128 N=64 K=16 with the bf16 gradient rows as A operand in TMEM and fp32 accumulators in
//     TMEM, warps 2..5 (one thread per row) read the accumulator, apply the ReLU mask (one bit per unit, written by the forward:
//     32 bytes per row and layer), pack to bf16, write the next A operand to TMEM and the gradient record to HBM.
//     Gradients with respect to the inputs (embedded points / directions) are not produced: the positional embedder has no
//     parameters (src/NeRF.cpp:4-39).
//
//  2. mlp_nerf_bwd_dw_kernel — dW_l = dY_l^T X_l and db_l = column sums of dY_l as ONE flat list of (unit, 64-row slab) work items
//     split evenly over the SMs.  A unit is a 128-wide output block of one weight matrix; both MMA operands are the record
//     regions as they lie in HBM (MN-major A and B, one bulk copy each per stage), accumulators stay in TMEM over a CTA's whole
//     range of a unit and leave as fp32 REDs into the caller's gradient tensors.  The 4 epilogue warps sum the columns of the
//     dY slabs from shared memory (bias gradients) while the tensor core works.
//
// bf16 operands, fp32 accumulation; parity tests/test_gpu_mlp_nerf.py (rel 1e-2 against the fp64 autograd of the oracle).
#include "mlp_nerf_layout.cuh"
#include "dw_units.cuh"
#include <algorithm>

namespace nrf {
namespace nerf_tc {

constexpr int kBwdThreads = 32 * 6;
// TMEM columns of the chain kernel: D fp32 [128 x 256] and TWO A buffers of bf16 [128 x 256] (128 columns each): step st reads
// A[st & 1] and its epilogue writes A[(st + 1) & 1] slab by slab while the MMAs of the later slabs still read the old operand.
// The 16-wide head operands live in columns no other operand needs at that time: [r g b 0..] at the start of A[0] (read by step
// 0, overwritten by step 1's output), [alpha 0..] at column 64 of A[1] (step 1's operand d_hv ends at 63; read by step 2).
constexpr uint32_t kBD = 0, kBA0 = 256, kBA1 = 384, kBRgb = kBA0, kBAlpha = kBA1 + 64;
__host__ __device__ constexpr uint32_t a_buf(int st) { return (st & 1) ? kBA1 : kBA0; }
constexpr int kSteps = 10;
// chain step -> the layer whose weights it multiplies: rgb, views, feature(+alpha), pts_linears 7..1
__host__ __device__ constexpr int step_layer(int st) { return st == 0 ? 11 : (st == 1 ? 10 : (st == 2 ? 8 : 10 - st)); }
__host__ __device__ constexpr int step_first_stage(int l) { return l == 5 ? 1 : 0; }        // stage 0 of layer 5 is the [pts] slab
__host__ __device__ constexpr int step_stages(int l) { return l == 11 ? 1 : 4; }

// The 38 weight stages of one tile in the order the chain consumes them, as (byte offset in the blob, bytes): a compile-time table in
// constant memory.  (Evaluating stage_offset(l, s) — nested loops over the layer table — per stage cost the producer thread ~2 000
// cycles per stage and was what the MMAs were waiting for: profiles/r1_mlp_nerf_bwd_chain_cycles.txt.)
constexpr int kChainStages = 38;
struct StageTable {
	int off[kChainStages], bytes[kChainStages];
};
constexpr StageTable make_chain_table()
{
	StageTable t{};
	int i = 0;
	for (int st = 0; st < kSteps; st++) {
		const int l = step_layer(st);
		for (int s = step_first_stage(l); s < step_first_stage(l) + step_stages(l); s++, i++) { t.off[i] = stage_offset(l, s); t.bytes[i] = stage_bytes(l, s); }
		if (st == 2) { t.off[i] = stage_offset(9, 0); t.bytes[i] = stage_bytes(9, 0); i++; }
	}
	return t;
}
__constant__ StageTable c_chain_table = make_chain_table();

// 6 x 32 KB: one and a half chain steps of weights in flight, so the stream keeps running through the epilogue tail of a step (with
// one step's worth the issuer waited ~500 cycles per stage for weights, profiles/r1_mlp_nerf_bwd_chain_cycles.txt)
constexpr int kChainRing = 6;
struct __align__(128) ChainSmem {
	uint8_t ring[kChainRing][kStageBytes];
	uint64_t full[kChainRing], empty[kChainRing];
	uint64_t a_ready, slab_ready[4];
	uint32_t tmem_base;
};

#ifdef NRF_PROFILE_CHAIN
// debug build only (NRF_NVCC_EXTRA=-DNRF_PROFILE_CHAIN): per-CTA cycle counters of the chain kernel, read back by nrf_debug_chain_profile
__device__ unsigned long long g_chain_prof[kNumSMs][8];
#define CH_T0() const long long t0__ = clock64()
#define CH_ADD(slot) g_chain_prof[blockIdx.x][slot] += static_cast<unsigned long long>(clock64() - t0__)
#else
#define CH_T0()
#define CH_ADD(slot)
#endif

// one 32-column accumulator chunk -> (* ReLU mask word of the forward: bit i / 16+i = low / high half of pair i) -> bf16 pairs
template <bool MASK>
__device__ __forceinline__ void grad_pack(const uint32_t (&acc)[32], uint32_t bits, uint32_t (&a16)[16])
{
#pragma unroll
	for (int i = 0; i < 16; i++) {
		uint32_t w = pack_bf16(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1]));
		if (MASK) w &= ((bits >> i) & 0x00010001u) * 0xFFFFu;
		a16[i] = w;
	}
}

// One chain step, slab by slab: the accumulator arrives as 64-column slabs (one per weight stage, each complete over K), so the
// epilogue of slab s runs while the tensor core still works on slabs s+1.. .  SLABS of the 4 slabs carry data (all 4 barriers are
// consumed to keep their phases in step).  bits: this row's 8 mask words of the step (32 bytes, fetched one step ahead).
template <int SLABS, bool MASK>
__device__ __forceinline__ void epilogue_grad(uint32_t t_lane, uint64_t* slab_ready, uint32_t parity, uint8_t* __restrict__ out_row, bool to_tmem,
	uint32_t a_next, const uint32_t (&bits)[8])
{
	uint32_t acc0[32], acc1[32], a16[16];
#pragma unroll
	for (int sl = 0; sl < 4; sl++) {
		{ CH_T0(); mbar_wait(&slab_ready[sl], parity); if (threadIdx.x == 64) CH_ADD(3); }
		if (sl >= SLABS) continue;
		CH_T0();
		fence_after();
		tmem_ld32(t_lane + kBD + 64 * sl, acc0);
		tmem_ld_wait_for(acc0);
		tmem_ld32(t_lane + kBD + 64 * sl + 32, acc1);
		grad_pack<MASK>(acc0, bits[2 * sl], a16);
		if (to_tmem) tmem_st16(t_lane + a_next + 32 * sl, a16);
		store_chunks(out_row, 8 * sl, a16);
		tmem_ld_wait_for(acc1);
		grad_pack<MASK>(acc1, bits[2 * sl + 1], a16);
		if (to_tmem) tmem_st16(t_lane + a_next + 32 * sl + 16, a16);
		store_chunks(out_row, 8 * sl + 4, a16);
		if (threadIdx.x == 64) CH_ADD(4);
	}
}

__device__ __forceinline__ void load_bits(const uint8_t* __restrict__ bits_row, bool wide, uint32_t (&b)[8])
{
	const uint4 lo = __ldg(reinterpret_cast<const uint4*>(bits_row));
	b[0] = lo.x; b[1] = lo.y; b[2] = lo.z; b[3] = lo.w;
	if (wide) {
		const uint4 hi = __ldg(reinterpret_cast<const uint4*>(bits_row) + 1);
		b[4] = hi.x; b[5] = hi.y; b[6] = hi.z; b[7] = hi.w;
	}
}

__global__ void __launch_bounds__(kBwdThreads, 1) mlp_nerf_bwd_chain_kernel(const uint8_t* __restrict__ blob, const uint8_t* __restrict__ saved,
	const float* __restrict__ grad_out, int64_t n, uint8_t* __restrict__ grads)
{
	extern __shared__ __align__(128) uint8_t smem_raw[];
	ChainSmem& sm = *reinterpret_cast<ChainSmem*>(smem_raw);
	const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;      // warp index the compiler can see is uniform
	const int64_t n_tiles = (n + 127) / 128;
	const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

	if (warp == 1) {
		if (lane == 0) {
			for (int s = 0; s < kChainRing; s++) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], 1); }
			mbar_init(&sm.a_ready, 4);
			for (int s = 0; s < 4; s++) mbar_init(&sm.slab_ready[s], 1);
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
		// ===== producer: 38 stages of the forward blob per tile, reverse layer order =====
		if (lane == 0) {
			uint32_t g = 0;
			auto push = [&](int off, uint32_t bytes) {
				const uint32_t slot = g % kChainRing, round = g / kChainRing;
				{ CH_T0(); mbar_wait(&sm.empty[slot], (round & 1u) ^ 1u); CH_ADD(7); }
				{
					CH_T0();
					mbar_expect_tx(&sm.full[slot], bytes);
					tma_bulk_g2s(sm.ring[slot], blob + off, bytes, &sm.full[slot]);
					CH_ADD(5);
				}
				g++;
			};
			for (int64_t t = 0; t < my_tiles; t++) {
#pragma unroll 1
				for (int i = 0; i < kChainStages; i++) push(c_chain_table.off[i], c_chain_table.bytes[i]);
			}
		}
	} else if (warp == 1) {
		// ===== MMA issuer: the whole warp runs the (warp-uniform) control flow, one elected lane issues =====
		const bool leader = elect_one();
		uint32_t g = 0, pa = 0;
		for (int64_t t = 0; t < my_tiles; t++) {
#pragma unroll 1
			for (int st = 0; st < kSteps; st++) {
				{ CH_T0(); mbar_wait(&sm.a_ready, pa); if (leader) CH_ADD(0); }
				pa ^= 1u;
				fence_after();
				const int l = step_layer(st);
				if (l == 11) {
					// d_hv = d_rgb * W_rgb: K = 16 (3 real), N = 128
					const uint32_t slot = g % kChainRing, round = g / kChainRing;
					mbar_wait(&sm.full[slot], round & 1u);
					fence_after();
					if (leader) {
						umma_ts(tmem + kBD, tmem + kBRgb, smem_desc(smem_u32(sm.ring[slot]), 128, 16 * 16), idesc(128, 128, true, 0, 1), 0u);
						umma_commit(&sm.empty[slot]);
						for (int s = 0; s < 4; s++) umma_commit(&sm.slab_ready[s]);
					}
					__syncwarp();
					g++;
				} else {
					const int n_out = layer_info(l).N;               // K of this product
					const uint32_t id = idesc(128, 64, true, 0, 1);
					for (int s = 0; s < 4; s++, g++) {
						const uint32_t slot = g % kChainRing, round = g / kChainRing;
						{ CH_T0(); mbar_wait(&sm.full[slot], round & 1u); if (leader) CH_ADD(1); }
						fence_after();
						CH_T0();
						// one descriptor per stage, then 16 (8) back-to-back MMAs whose operands differ by constants: the issuing thread
						// must not spend more than the 32 cycles an N = 64 MMA takes on each of them
						const uint64_t b0 = smem_desc(smem_u32(sm.ring[slot]), 128, n_out * 16);
						const uint32_t d = tmem + kBD + 64 * s, a0 = tmem + a_buf(st);
						if (leader) {
							if (n_out == 256) issue_k<16>(d, a0, b0, id, 0u);
							else issue_k<8>(d, a0, b0, id, 0u);
							umma_commit(&sm.empty[slot]);
							if (st != 2) umma_commit(&sm.slab_ready[s]);     // this 64-column slab of D is complete
							CH_ADD(2);
						}
						__syncwarp();
					}
					if (st == 2) {
						// + d_alpha * W_alpha over all 256 columns: K = 16 (1 real)
						const uint32_t slot = g % kChainRing, round = g / kChainRing;
						mbar_wait(&sm.full[slot], round & 1u);
						fence_after();
						if (leader) {
							umma_ts(tmem + kBD, tmem + kBAlpha, smem_desc(smem_u32(sm.ring[slot]), 128, 16 * 16), idesc(128, 256, true, 0, 1), 1u);
							umma_commit(&sm.empty[slot]);
							for (int s = 0; s < 4; s++) umma_commit(&sm.slab_ready[s]);
						}
						__syncwarp();
						g++;
					}
				}
			}
		}
	} else {
		// ===== epilogue warps: one thread per row =====
		const int q = warp & 3;
		const int row = (q << 5) | lane;
		const uint32_t t_lane = tmem + (static_cast<uint32_t>(q << 5) << 16);
		uint32_t pd = 0;
#ifdef NRF_PROFILE_CHAIN
		const long long t_start = clock64();
#endif
		for (int64_t t = 0; t < my_tiles; t++) {
			const int64_t tile = blockIdx.x + t * gridDim.x;
			const int64_t r = tile * 128 + row;
			const uint8_t* const rec_s = saved + tile * kSaveTile;
			uint8_t* const rec_g = grads + tile * kGradTile;
			uint32_t bits[8];
			{
				float4 g4 = make_float4(0.f, 0.f, 0.f, 0.f);
				if (r < n) g4 = __ldg(reinterpret_cast<const float4*>(grad_out) + r);
				uint32_t a16[16];
#pragma unroll
				for (int i = 0; i < 16; i++) a16[i] = 0u;
				a16[0] = pack_bf16(g4.x, g4.y);
				a16[1] = pack_bf16(g4.z, 0.f);
				tmem_st16(t_lane + kBRgb, a16);          // K = 16 operand [r g b 0..]
				uint8_t* o = rec_g + kGradOut + chunk_offset(16, row, 0);
				*reinterpret_cast<uint4*>(o) = make_uint4(a16[0], pack_bf16(g4.z, g4.w), 0u, 0u);
				a16[0] = pack_bf16(g4.w, 0.f);
				a16[1] = 0u;
				tmem_st16(t_lane + kBAlpha, a16);        // K = 16 operand [alpha 0..]
				*reinterpret_cast<uint4*>(o + 1024) = make_uint4(0u, 0u, 0u, 0u);
			}
			load_bits(rec_s + bits_offset(0, row), false, bits);
			publish(&sm.a_ready, lane);

#pragma unroll 1
			for (int st = 0; st < kSteps; st++) {
				if (st == 0) {
					epilogue_grad<2, true>(t_lane, sm.slab_ready, pd, rec_g + kGradHv + chunk_offset(128, row, 0), true, a_buf(1), bits);
				} else if (st == 1) {
					epilogue_grad<4, false>(t_lane, sm.slab_ready, pd, rec_g + kGradFeat + chunk_offset(256, row, 0), true, a_buf(2), bits);
				} else {
					const int l = st == 2 ? 8 : 10 - st;         // the activation h_l whose ReLU is undone; the result is dY_{l-1}
					epilogue_grad<4, true>(t_lane, sm.slab_ready, pd, rec_g + grad_y(l - 1) + chunk_offset(256, row, 0), st + 1 < kSteps, a_buf(st + 1), bits);
				}
				pd ^= 1u;
				if (st + 1 < kSteps) {
					// the 32 mask bytes of the next step (h_8 after step 1, then h_7 .. h_1), requested before that step's MMAs are even issued
					CH_T0();
					if (st >= 1) load_bits(rec_s + bits_offset(st == 1 ? 8 : (st == 2 ? 8 : 10 - st) - 1, row), true, bits);
					publish(&sm.a_ready, lane);
				}
			}
		}
#ifdef NRF_PROFILE_CHAIN
		if (threadIdx.x == 64) g_chain_prof[blockIdx.x][6] += static_cast<unsigned long long>(clock64() - t_start);
#endif
	}

	fence_before();
	__syncthreads();
	if (warp == 1) {
		fence_after();
		tmem_free_all(tmem);
	}
}

// ---- weight gradients --------------------------------------------------------------------------------------------------
// A unit is one weight matrix (or one column block of it): D[M = columns of the A region (128 or 256), N] = A^T B summed over rows.
// M = 256 runs as two M = 128 MMAs on the same B slab, so a dY slab and an activation slab are each read from HBM once per unit.
constexpr int kDwRing = 3;
constexpr int kDwStageBytes = 256 * 64 * 2 + 256 * 64 * 2;         // A: up to 256 columns x 64 rows, B: up to 256 columns x 64 rows
constexpr int kDwAOff = 0, kDwBOff = 256 * 64 * 2;
using dw::Unit;
using dw::UnitTable;
using dw::kMaxUnits;

struct __align__(128) DwSmem {
	uint8_t ring[kDwRing][kDwStageBytes];
	uint64_t full[kDwRing], empty[kDwRing];
	uint64_t d_ready, d_free;
	uint32_t tmem_base;
};

#ifdef NRF_PROFILE_DW
// debug build only (NRF_NVCC_EXTRA=-DNRF_PROFILE_DW): per-CTA cycle counters of the dW kernel, read back by nrf_debug_dw_profile
__device__ unsigned long long g_dw_prof[kNumSMs][8];
#define DW_T0() const long long t0__ = clock64()
#define DW_ADD(slot) g_dw_prof[blockIdx.x][slot] += static_cast<unsigned long long>(clock64() - t0__)
__device__ __forceinline__ void g_prof_items(long long n) { g_dw_prof[blockIdx.x][7] += static_cast<unsigned long long>(n); }
#else
__device__ __forceinline__ void g_prof_items(long long) {}
#define DW_T0()
#define DW_ADD(slot)
#endif

__device__ __forceinline__ int64_t clamp_items(int64_t x, int64_t h) { return x < 0 ? 0 : (x > h ? h : x); }
// relative time of one 64-row slab of a unit (measured per CTA with clock64, profiles/r1_mlp_nerf_bwd_dw_balance.txt): bytes moved for
// the wide products, a latency floor (three slabs in flight) for the narrow ones
__host__ __device__ __forceinline__ int64_t unit_cost(int a_cols, int b_cols)
{
	const int c = b_cols >= 64 ? a_cols + (b_cols > 160 ? b_cols : 160) : a_cols + b_cols;
	return c > 272 ? c : 272;
}

__global__ void __launch_bounds__(kBwdThreads, 1) mlp_nerf_bwd_dw_kernel(const __grid_constant__ UnitTable T, const uint8_t* __restrict__ saved,
	const uint8_t* __restrict__ grads, int64_t n_tiles)
{
	extern __shared__ __align__(128) uint8_t smem_raw[];
	DwSmem& sm = *reinterpret_cast<DwSmem*>(smem_raw);
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int64_t H = 2 * n_tiles;                                   // 64-row slabs per unit
	int64_t total = 0;
	for (int u = 0; u < T.count; u++) total += H * unit_cost(T.u[u].a_cols, T.u[u].b_cols);
	const int64_t lo_cost = total / gridDim.x * blockIdx.x + (total % gridDim.x) * blockIdx.x / gridDim.x;
	const int64_t hi_cost = total / gridDim.x * (blockIdx.x + 1) + (total % gridDim.x) * (blockIdx.x + 1) / gridDim.x;

	if (warp == 1) {
		if (lane == 0) {
			for (int s = 0; s < kDwRing; s++) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], 5); }
			mbar_init(&sm.d_ready, 1);
			mbar_init(&sm.d_free, 4);
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
		// ===== producer: one bulk copy per operand and slab =====
		if (lane == 0) {
			uint32_t g = 0;
			int64_t cum = 0;
			for (int u = 0; u < T.count; u++) {
				const Unit& U = T.u[u];
				const int64_t c = unit_cost(U.a_cols, U.b_cols);
				const int64_t lo = clamp_items((lo_cost - cum) / c, H), hi = clamp_items((hi_cost - cum) / c, H);
				cum += H * c;
				const uint8_t* a_base = (U.a_src ? saved : grads) + U.a_off;
				const uint8_t* b_base = (U.b_src ? saved : grads) + U.b_off;
				const int64_t a_tile = U.a_src ? T.save_tile : T.grad_tile, b_tile = U.b_src ? T.save_tile : T.grad_tile;
				const uint32_t a_bytes = U.a_cols * 128, b_bytes = U.b_cols * 128;      // one 64-row half of the operand's columns
				const uint32_t a_half = U.a_half ? U.a_half : a_bytes, b_half = U.b_half ? U.b_half : b_bytes;   // distance between the halves (region width x 128)
				for (int64_t i = lo; i < hi; i++, g++) {
					const uint32_t slot = g % kDwRing, round = g / kDwRing;
					{ DW_T0(); mbar_wait(&sm.empty[slot], (round & 1u) ^ 1u); DW_ADD(2); }
					mbar_expect_tx(&sm.full[slot], a_bytes + b_bytes);
					tma_bulk_g2s(sm.ring[slot] + kDwAOff, a_base + (i >> 1) * a_tile + (i & 1) * a_half, a_bytes, &sm.full[slot]);
					tma_bulk_g2s(sm.ring[slot] + kDwBOff, b_base + (i >> 1) * b_tile + (i & 1) * b_half, b_bytes, &sm.full[slot]);
				}
			}
		}
	} else if (warp == 1) {
		// ===== MMA issuer: D[m block][128, N] += A^T B over the 64 rows of a slab: 4 K steps x (1 or 2) M blocks =====
		if (lane == 0) {
			uint32_t g = 0, seg = 0;
			int64_t cum = 0;
			for (int u = 0; u < T.count; u++) {
				const Unit& U = T.u[u];
				const int64_t c = unit_cost(U.a_cols, U.b_cols);
				const int64_t lo = clamp_items((lo_cost - cum) / c, H), hi = clamp_items((hi_cost - cum) / c, H);
				cum += H * c;
				if (hi <= lo) continue;
				{ DW_T0(); mbar_wait(&sm.d_free, (seg & 1u) ^ 1u); DW_ADD(1); }         // the accumulators of the previous segment have been read out
				fence_after();
				// both operands bf16, MN-major.  (A and B of a tcgen05.mma kind::f16 must carry the SAME 16-bit format: an instruction descriptor that
				// mixes bf16 gradient rows with fp16 activation rows raises an illegal-instruction fault on B200, gpurun_out/r2i.)
				const uint32_t id = idesc(128, U.b_cols, true, 1, 1);
				const int mblocks = U.a_cols / 128;
				for (int64_t i = lo; i < hi; i++, g++) {
					const uint32_t slot = g % kDwRing, round = g / kDwRing;
					{ DW_T0(); mbar_wait(&sm.full[slot], round & 1u); DW_ADD(0); }
					fence_after();
					const uint32_t saddr = smem_u32(sm.ring[slot]);
					const uint64_t a0 = smem_desc(saddr + kDwAOff, 128, 1024), b0 = smem_desc(saddr + kDwBOff, 128, 1024);
					const uint32_t acc = i > lo ? 1u : 0u;
					if (mblocks == 2) {
#pragma unroll
						for (int j = 0; j < 4; j++) {
							umma_ss(tmem, a0 + static_cast<uint64_t>(16 * j), b0 + static_cast<uint64_t>(16 * j), id, j ? 1u : acc);
							umma_ss(tmem + 256, a0 + static_cast<uint64_t>(1024 + 16 * j), b0 + static_cast<uint64_t>(16 * j), id, j ? 1u : acc);
						}
					} else {
#pragma unroll
						for (int j = 0; j < 4; j++) umma_ss(tmem, a0 + static_cast<uint64_t>(16 * j), b0 + static_cast<uint64_t>(16 * j), id, j ? 1u : acc);
					}
					umma_commit(&sm.empty[slot]);
				}
				umma_commit(&sm.d_ready);
				seg++;
			}
		}
	} else {
		// ===== epilogue warps: bias column sums while the slabs stream, then the accumulator flush =====
		const int q = warp & 3;
		const uint32_t t_lane = tmem + (static_cast<uint32_t>(q << 5) << 16);
		uint32_t g = 0, seg = 0;
		int64_t cum = 0;
#ifdef NRF_PROFILE_DW
		const long long t_start = clock64();
		unsigned long long g_start;
		asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_start));
#endif
		for (int u = 0; u < T.count; u++) {
			const Unit& U = T.u[u];
			const int64_t c = unit_cost(U.a_cols, U.b_cols);
			const int64_t lo = clamp_items((lo_cost - cum) / c, H), hi = clamp_items((hi_cost - cum) / c, H);
			cum += H * c;
			if (hi <= lo) continue;
			float bs[8][8];
#pragma unroll
			for (int a = 0; a < 8; a++)
#pragma unroll
				for (int e = 0; e < 8; e++) bs[a][e] = 0.f;
			const bool sum_a = U.bias_mode == 1, sum_b = U.bias_mode == 2 && q == 0;
			const int per_warp = U.a_cols / 32;          // column chunks of the A slab per warp: 8 (256 columns) or 4
			for (int64_t i = lo; i < hi; i++, g++) {
				const uint32_t slot = g % kDwRing, round = g / kDwRing;
				mbar_wait(&sm.full[slot], round & 1u);
				if (sum_a || sum_b) {
					// warp q owns column chunks per_warp*q .. of the A slab (or chunk 0 of the B slab); lanes take rows lane, lane + 32
					const uint8_t* base = sm.ring[slot] + (sum_a ? kDwAOff + (per_warp * q) * 1024 : kDwBOff);
#pragma unroll
					for (int a = 0; a < 8; a++) {
						if (a < (sum_a ? per_warp : 1)) {
#pragma unroll
							for (int h = 0; h < 2; h++) {
								const uint4 v = *reinterpret_cast<const uint4*>(base + a * 1024 + (lane + 32 * h) * 16);
								const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
								for (int e = 0; e < 4; e++) {
									bs[a][2 * e] += __uint_as_float(w[e] << 16);
									bs[a][2 * e + 1] += __uint_as_float(w[e] & 0xFFFF0000u);
								}
							}
						}
					}
				}
				__syncwarp();
				if (lane == 0) mbar_arrive(&sm.empty[slot]);
			}
			// ---- flush ----
			DW_T0();
			if (sum_a || sum_b) {
#pragma unroll
				for (int a = 0; a < 8; a++)
#pragma unroll
					for (int e = 0; e < 8; e++) {
						const float s = warp_sum(bs[a][e]);
						if (lane == 0) {
							if (sum_a) { if (a < per_warp) atomicAdd(U.bias + 8 * (per_warp * q + a) + e, s); }
							else if (a == 0 && e < 3) atomicAdd(U.bias + e, s);
							else if (a == 0 && e == 3) atomicAdd(U.bias2, s);
						}
					}
			}
			mbar_wait(&sm.d_ready, seg & 1u);
			fence_after();
			if (warp == 2 && lane == 0) DW_ADD(5);
			for (int mb = 0; mb < U.a_cols / 128; mb++) {
				const int m = 128 * mb + 32 * q + lane;
				for (int c0 = 0; c0 < U.b_cols; c0 += 16) {
					uint32_t d16[16];
					tmem_ld16(t_lane + 256 * mb + c0, d16);
					tmem_ld_wait();
					float* row = U.out + static_cast<int64_t>(m) * U.stride_m;
					if (U.stride_n == 1 && c0 >= U.n_lo && c0 + 16 <= U.n_hi && ((reinterpret_cast<uintptr_t>(row + (c0 - U.n_lo))) & 15) == 0) {
						// 16-byte vector REDs: the L2 atomic units are bound per operation, not per byte
#pragma unroll
						for (int j = 0; j < 16; j += 4)
							asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(row + (c0 - U.n_lo) + j), "f"(__uint_as_float(d16[j])),
								"f"(__uint_as_float(d16[j + 1])), "f"(__uint_as_float(d16[j + 2])), "f"(__uint_as_float(d16[j + 3])) : "memory");
					} else {
#pragma unroll
						for (int j = 0; j < 16; j++) {
							const int nn = c0 + j;
							if (nn >= U.n_lo && nn < U.n_hi) atomicAdd(row + static_cast<int64_t>(nn - U.n_lo) * U.stride_n, __uint_as_float(d16[j]));
							else if (U.out2 != nullptr && nn >= U.n2_lo && nn < U.n2_hi)
								atomicAdd(U.out2 + static_cast<int64_t>(m) * U.stride_m + static_cast<int64_t>(nn - U.n2_lo) * U.stride_n, __uint_as_float(d16[j]));
						}
					}
				}
			}
			fence_before();
			__syncwarp();
			if (lane == 0) mbar_arrive(&sm.d_free);
			if (warp == 2 && lane == 0) { DW_ADD(6); g_prof_items(hi - lo); }
			seg++;
		}
#ifdef NRF_PROFILE_DW
		if (warp == 2 && lane == 0) {
			unsigned long long g_end;
			asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_end));
			g_dw_prof[blockIdx.x][3] += static_cast<unsigned long long>(clock64() - t_start);       // whole kernel, cycles
			g_dw_prof[blockIdx.x][4] += g_end - g_start;                                          // whole kernel, ns
		}
#endif
	}

	fence_before();
	__syncthreads();
	if (warp == 1) {
		fence_after();
		tmem_free_all(tmem);
	}
}

static Unit make_unit(int a_src, int a_region, int a_cols, int b_src, int b_region, int b_cols, int n_lo, int n_hi, int stride_m, int stride_n, float* out,
	int bias_mode = 0, float* bias = nullptr, float* bias2 = nullptr)
{
	Unit u{};
	u.a_src = a_src; u.a_off = a_region; u.a_cols = a_cols;
	u.b_src = b_src; u.b_off = b_region; u.b_cols = b_cols;
	u.n_lo = n_lo; u.n_hi = n_hi; u.stride_m = stride_m; u.stride_n = stride_n;
	u.bias_mode = bias_mode; u.out = out; u.bias = bias; u.bias2 = bias2;
	return u;
}

static void build_units(const Grads& g, UnitTable& T)
{
	int c = 0;
	for (int l = 0; l < 8; l++) {
		const int ld = l == 0 ? kInPts : (l == 5 ? kW + kInPts : kW);
		if (l == 0) {
			T.u[c++] = make_unit(0, grad_y(0), 256, 1, kSavePts, 64, 0, kInPts, ld, 1, g.w[0], 1, g.b[0]);
		} else if (l == 5) {                                                      // [pts | h5]
			T.u[c++] = make_unit(0, grad_y(5), 256, 1, kSavePts, 64, 0, kInPts, ld, 1, g.w[5]);
			T.u[c++] = make_unit(0, grad_y(5), 256, 1, save_h(5), 256, 0, 256, ld, 1, g.w[5] + kInPts, 1, g.b[5]);
		} else {
			T.u[c++] = make_unit(0, grad_y(l), 256, 1, save_h(l), 256, 0, 256, ld, 1, g.w[l], 1, g.b[l]);
		}
	}
	T.u[c++] = make_unit(0, kGradFeat, 256, 1, save_h(8), 256, 0, 256, kW, 1, g.w[8], 1, g.b[8]);                          // feature_linear
	T.u[c++] = make_unit(0, kGradHv, 128, 1, kSaveFeat, 256, 0, 256, kW + kInViews, 1, g.w[10], 1, g.b[10]);               // views_linears[0]: [feature |
	T.u[c++] = make_unit(0, kGradHv, 128, 1, kSaveViews, 32, 0, kInViews, kW + kInViews, 1, g.w[10] + kW);                 //                     views]
	// heads, roles swapped (M = input index): rgb_linear [3,128] from hv, alpha_linear [1,256] from h8; their biases from dOut
	T.u[c++] = make_unit(1, kSaveHv, 128, 0, kGradOut, 16, 0, 3, 1, kW / 2, g.w[11], 2, g.b[11], g.b[9]);
	T.u[c++] = make_unit(1, save_h(8), 256, 0, kGradOut, 16, 3, 4, 1, kW, g.w[9]);
	T.count = c;
}

}  // namespace nerf_tc

namespace dw {
int launch_dw_units(const UnitTable& T, const void* saved, const void* grads, int64_t n_tiles, nrf_stream stream)
{
	using namespace nerf_tc;
	const int64_t items = 2 * n_tiles * T.count;
	const int blocks = static_cast<int>(std::min<int64_t>(items, kNumSMs));
	const int smem = static_cast<int>(sizeof(DwSmem)) + 128;
	NRF_CUDA(cudaFuncSetAttribute(mlp_nerf_bwd_dw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
	mlp_nerf_bwd_dw_kernel<<<blocks, kBwdThreads, smem, as_stream(stream)>>>(T, reinterpret_cast<const uint8_t*>(saved), reinterpret_cast<const uint8_t*>(grads), n_tiles);
	NRF_CHECK_LAUNCH("mlp_nerf_bwd_dw_kernel");
	return NRF_OK;
}
}  // namespace dw
}  // namespace nrf

using namespace nrf;
using namespace nrf::nerf_tc;

extern "C" {

int64_t nrf_mlp_nerf_bwd_workspace_bytes(const nrf_mlp_nerf_shape* shape, int64_t n)
{
	if (nerf_tc::check_shape(shape) || n < 0) return -1;
	return ((n + 127) / 128) * static_cast<int64_t>(kGradTile);
}

int nrf_mlp_nerf_bwd(const nrf_mlp_nerf_shape* shape, const void* packed_train, const void* saved, const float* grad_out, int64_t n, void* workspace,
                     const nrf_mlp_nerf_grads* grads, nrf_stream stream)
{
	if (int rc = nerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(n >= 0, "negative n");
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(packed_train && saved && grad_out && workspace && grads, "null pointer");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(packed_train) & 127) == 0 && (reinterpret_cast<uintptr_t>(saved) & 127) == 0 &&
		(reinterpret_cast<uintptr_t>(workspace) & 127) == 0 && (reinterpret_cast<uintptr_t>(grad_out) & 15) == 0,
		"packed / saved / workspace must be 128-byte, grad_out 16-byte aligned");
	Grads g;
	for (int i = 0; i < 8; i++) { g.w[i] = grads->pts_w[i]; g.b[i] = grads->pts_b[i]; }
	g.w[8] = grads->feature_w; g.b[8] = grads->feature_b;
	g.w[9] = grads->alpha_w; g.b[9] = grads->alpha_b;
	g.w[10] = grads->views_w; g.b[10] = grads->views_b;
	g.w[11] = grads->rgb_w; g.b[11] = grads->rgb_b;
	for (int i = 0; i < kLayers; i++) NRF_REQUIRE(g.w[i] && g.b[i], "null gradient pointer");
	const int64_t tiles = (n + 127) / 128;
	{
		const int blocks = static_cast<int>(std::min<int64_t>(tiles, kNumSMs));
		const int smem = static_cast<int>(sizeof(ChainSmem)) + 128;
		NRF_CUDA(cudaFuncSetAttribute(mlp_nerf_bwd_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
		mlp_nerf_bwd_chain_kernel<<<blocks, kBwdThreads, smem, as_stream(stream)>>>(reinterpret_cast<const uint8_t*>(packed_train),
			reinterpret_cast<const uint8_t*>(saved), grad_out, n, reinterpret_cast<uint8_t*>(workspace));
		NRF_CHECK_LAUNCH("mlp_nerf_bwd_chain_kernel");
	}
	{
		UnitTable T{};
		build_units(g, T);
		T.save_tile = kSaveTile;
		T.grad_tile = kGradTile;
		if (int rc = dw::launch_dw_units(T, saved, workspace, tiles, stream)) return rc;
	}
	return NRF_OK;
}

#ifdef NRF_PROFILE_CHAIN
/* debug builds only: [148][8] cycle counters {issuer waits a_ready, issuer waits full, issuer issue+commit, epilogue waits slab_ready,
 * epilogue work, mask fetch + publish, epilogue warp total, producer waits empty}; clears them */
int nrf_debug_chain_profile(unsigned long long* host_out)
{
	NRF_CUDA(cudaDeviceSynchronize());
	NRF_CUDA(cudaMemcpyFromSymbol(host_out, g_chain_prof, sizeof(unsigned long long) * kNumSMs * 8));
	static unsigned long long zeros[kNumSMs * 8] = {};
	NRF_CUDA(cudaMemcpyToSymbol(g_chain_prof, zeros, sizeof(zeros)));
	return NRF_OK;
}
#endif

#ifdef NRF_PROFILE_DW
/* debug builds only: [148][8] cycle counters {issuer waits full, issuer waits d_free, producer waits empty, epilogue waits full, epilogue sums,
 * epilogue waits d_ready (incl. bias flush), flush incl. d_ready wait, items}; clears them */
int nrf_debug_dw_profile(unsigned long long* host_out)
{
	NRF_CUDA(cudaDeviceSynchronize());
	NRF_CUDA(cudaMemcpyFromSymbol(host_out, g_dw_prof, sizeof(unsigned long long) * kNumSMs * 8));
	static unsigned long long zeros[kNumSMs * 8] = {};
	NRF_CUDA(cudaMemcpyToSymbol(g_dw_prof, zeros, sizeof(zeros)));
	return NRF_OK;
}
#endif

}
