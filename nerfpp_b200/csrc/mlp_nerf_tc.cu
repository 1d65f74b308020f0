// Fused classic NeRF MLP forward (8 x 256, skip at layer 4, view branch) on tcgen05 / TMEM / TMA for sm_100a.
//
// Replaces NeRFImpl::forward (reference src/NeRF.cpp:92-126: 11 cuBLAS SGEMMs + bias/ReLU/cat kernels, every [N,256] fp32
// activation round-tripping HBM, SURVEY §8a-a7) for inference: x [N, 63+27] fp32 (the positional embeddings of points and view
// directions, src/NeRFRenderer.h:182) -> [N,4] = [rgb logits, alpha] (src/NeRF.cpp:120).
//
// Mapping (one persistent CTA per SM, one 128-point tile in flight):
//   * activations never leave the SM: the A operand of every layer lives in TENSOR MEMORY as fp16 (TMEM columns 272..447:
//     [pts 64 | h 256 | views 32] so that the skip layer reads [pts | h] and the view layer [feature | views] as ONE contiguous
//     K range), accumulators D are fp32 in TMEM columns 0..255 (+16 for the 1- and 3-wide heads);
//   * weights stream from L2 through a 4-deep ring of 32 KB shared-memory stages (one 64-wide K slab of a layer per stage,
//     pre-packed by nrf_mlp_nerf_pack as UMMA K-major core matrices, so a stage is ONE contiguous TMA bulk copy);
//     41 stages = 1.2 MB per tile, the same sequence for every tile;
//   * warp 0 / lane 0 produces stages (mbarrier expect_tx + cp.async.bulk), warp 1 / lane 0 issues tcgen05.mma M=128, N<=256,
//     K=16 per instruction and releases each stage with tcgen05.commit, warps 2..5 are the epilogue: one thread per row reads its
//     accumulator row with tcgen05.ld, adds the bias (shared memory), applies ReLU, packs to fp16 and writes the next layer's A
//     operand back to TMEM with tcgen05.st.
// fp16 operands, fp32 accumulation: <= 1e-2 relative to the fp32 reference (tests/test_gpu_mlp_nerf.py).
#include "mlp_nerf_layout.cuh"
#include <utility>

namespace nrf {
namespace nerf_tc {

constexpr int kThreads = 32 * 6;
constexpr int kStagePitch = 98;      // 16-bit elements per staged row (96 used): 49 words, odd, so the per-row accesses are conflict-free

// padded logical weight Wp_l(n, k) in the kernel's A-operand order
__device__ __forceinline__ float wp(const Weights& p, int l, int n, int k)
{
	switch (l) {
		case 0: return k < kInPts ? p.w[0][n * kInPts + k] : 0.f;
		case 5: return k < kInPts ? p.w[5][n * (kW + kInPts) + k] : (k < 64 ? 0.f : p.w[5][n * (kW + kInPts) + kInPts + (k - 64)]);   // [pts | h]
		case 9: return n < 1 ? p.w[9][k] : 0.f;
		case 10: return k < kW + kInViews ? p.w[10][n * (kW + kInViews) + k] : 0.f;                                                   // [feature | views]
		case 11: return n < 3 ? p.w[11][n * (kW / 2) + k] : 0.f;
		default: return p.w[l][n * kW + k];
	}
}

__global__ void __launch_bounds__(256) nerf_pack_kernel(Weights p, uint32_t* __restrict__ blob, bool bf16)
{
	const int w = blockIdx.x * blockDim.x + threadIdx.x;
	if (w >= kPackedBytes / 4) return;
	if (w >= kWeightBytes / 4) {
		const int i = w - kWeightBytes / 4;
		int l = 0;
		while (l + 1 < kLayers && i >= bias_offset(l + 1)) l++;
		const int n = i - bias_offset(l);
		const int real = l == 9 ? 1 : (l == 11 ? 3 : layer_info(l).N);
		reinterpret_cast<float*>(blob)[w] = n < real ? p.b[l][n] : 0.f;
		return;
	}
	int l = 0;
	while (l + 1 < kLayers && w * 4 >= layer_offset(l + 1)) l++;
	int q = w - layer_offset(l) / 4, s = 0, k_off = 0;
	while (q >= stage_bytes(l, s) / 4) { q -= stage_bytes(l, s) / 4; k_off += stage_k(l, s); s++; }
	const auto [n, k] = stage_word(q, layer_info(l).N, k_off);
	blob[w] = bf16 ? pack_bf16(wp(p, l, n, k), wp(p, l, n, k + 1)) : pack_f16(wp(p, l, n, k), wp(p, l, n, k + 1));
}

// the 41 weight stages of one tile as (byte offset, bytes): compile-time table in constant memory, so that the producer thread does not
// walk the layer table (nested constexpr loops evaluated at run time) for every stage
constexpr int kFwdStages = 41;
struct FwdStageTable {
	int off[kFwdStages], bytes[kFwdStages];
};
constexpr FwdStageTable make_fwd_table()
{
	FwdStageTable t{};
	int i = 0;
	for (int l = 0; l < kLayers; l++)
		for (int s = 0; s < layer_stages(l); s++, i++) { t.off[i] = stage_offset(l, s); t.bytes[i] = stage_bytes(l, s); }
	return t;
}
static_assert(make_fwd_table().off[kFwdStages - 1] + make_fwd_table().bytes[kFwdStages - 1] == kWeightBytes, "stage table does not cover the blob");
__constant__ FwdStageTable c_fwd_table = make_fwd_table();

struct __align__(128) Smem {
	uint8_t ring[kRing][kStageBytes];
	float bias[kBiasFloats];
	uint16_t stage[128 * kStagePitch];      // RAW input mode: one row of 64 + 32 embedding channels per thread (25 KB)
	uint64_t full[kRing], empty[kRing];
	uint64_t a_ready, d_ready;
	uint32_t tmem_base;
};

// epilogue of a 32-column accumulator chunk: + bias, optional ReLU, pack to 16 fp16 pairs
template <bool RELU, bool BF16>
__device__ __forceinline__ void bias_act_pack(const uint32_t (&acc)[32], const float* __restrict__ bias, uint32_t (&out)[16])
{
#pragma unroll
	for (int i = 0; i < 8; i++) {
		const float4 b = *reinterpret_cast<const float4*>(bias + 4 * i);
		const float v0 = __uint_as_float(acc[4 * i]) + b.x, v1 = __uint_as_float(acc[4 * i + 1]) + b.y;
		const float v2 = __uint_as_float(acc[4 * i + 2]) + b.z, v3 = __uint_as_float(acc[4 * i + 3]) + b.w;
		if (BF16) {
			out[2 * i] = RELU ? pack_bf16_relu(v0, v1) : pack_bf16(v0, v1);
			out[2 * i + 1] = RELU ? pack_bf16_relu(v2, v3) : pack_bf16(v2, v3);
		} else {
			out[2 * i] = RELU ? pack_f16_relu(v0, v1) : pack_f16(v0, v1);
			out[2 * i + 1] = RELU ? pack_f16_relu(v2, v3) : pack_f16(v2, v3);
		}
	}
}

// ReLU mask word of 32 packed columns: bit i / 16+i = low / high half of pair i is non-zero (values are >= 0 after ReLU)
__device__ __forceinline__ uint32_t relu_bits(const uint32_t (&a16)[16])
{
	uint32_t bits = 0;
#pragma unroll
	for (int i = 0; i < 16; i++) bits += __vminu2(a16[i], 0x00010001u) << i;
	return bits;
}

// D[:, 0 .. 32*CHUNKS) + bias -> (ReLU) -> fp16 -> the h columns, one thread per row.  The tcgen05.ld of chunk c+1 is in flight while
// chunk c is converted and stored (two register buffers), so the TMEM read latency is paid once, not once per chunk.  TRAIN: the packed
// columns also go to the scratch record (save_row) and, RELU, their mask words to bits_row.
template <int CHUNKS, bool RELU, bool TRAIN>
__device__ __forceinline__ void epilogue_to_h(uint32_t t_lane, const float* __restrict__ bias, uint8_t* __restrict__ save_row, uint8_t* __restrict__ bits_row)
{
	uint32_t acc0[32], acc1[32], a16[16];
	uint32_t bw[CHUNKS];
	tmem_ld32(t_lane + kColD, acc0);
#pragma unroll
	for (int c = 0; c < CHUNKS; c += 2) {
		tmem_ld_wait_for(acc0);
		if (c + 1 < CHUNKS) tmem_ld32(t_lane + kColD + 32 * (c + 1), acc1);
		bias_act_pack<RELU, TRAIN>(acc0, bias + 32 * c, a16);
		tmem_st16(t_lane + kColH + 16 * c, a16);
		if (TRAIN) store_chunks(save_row, 4 * c, a16);
		if (TRAIN && RELU) bw[c] = relu_bits(a16);
		if (c + 1 < CHUNKS) {
			tmem_ld_wait_for(acc1);
			if (c + 2 < CHUNKS) tmem_ld32(t_lane + kColD + 32 * (c + 2), acc0);
			bias_act_pack<RELU, TRAIN>(acc1, bias + 32 * (c + 1), a16);
			tmem_st16(t_lane + kColH + 16 * (c + 1), a16);
			if (TRAIN) store_chunks(save_row, 4 * (c + 1), a16);
			if (TRAIN && RELU) bw[c + 1] = relu_bits(a16);
		}
	}
	if (TRAIN && RELU) {
#pragma unroll
		for (int c = 0; c < CHUNKS; c += 4) *reinterpret_cast<uint4*>(bits_row + 4 * c) = make_uint4(bw[c], bw[c + 1], bw[c + 2], bw[c + 3]);
	}
}

// groups of layers that share one A operand and one epilogue: {0} {1} {2} {3} {4} {5} {6} {7} {8,9} {10} {11}
constexpr int kGroups = 11;
__host__ __device__ constexpr int group_first(int g) { return g <= 8 ? g : g + 1; }
__host__ __device__ constexpr int group_count(int g) { return g == 8 ? 2 : 1; }

// TRAIN: bf16 operands (the exponent range survives Xavier(0.1) initialisation, src/LibTorchTraining/Trainable.h:43, where fp16
// activations of the deep layers flush to zero) and every layer's input is stored to the scratch records of mlp_nerf_layout.cuh
// RAW: x is the sample positions [N,3] and the positional embedding (EmbedderImpl::forward, src/NeRF.cpp:22-39: [x, sin(f0 x), cos(f0 x), ..],
// same fp32 product and libdevice sinf / cosf as nrf_posenc_fwd, hence bit-identical operands) is evaluated by the thread that owns the row,
// directions are read per RAY (row / samples_per_ray; the reference expands them per sample, src/NeRFRenderer.h:179-181): the [N,63] / [N,27]
// embeddings and their [N,90] concatenation (src/NeRFRenderer.h:182) never exist in memory.
struct RawInput {
	const float* dirs;       // [R,3]
	int samples_per_ray;
	float fp[10], fv[4];     // frequency bands of the two embedders
};


// x(3), then per band sin(3), cos(3) of one 3-vector, rounded to the operand type and written to this thread's staging row.  The band loop
// is NOT unrolled on purpose: 84 inlined sinf / cosf bodies per thread (~5 000 SASS instructions) pushed the kernel out of the instruction
// cache and cost more than the whole MLP tile.
template <bool BF16>
__device__ __forceinline__ void posenc_stage(const float (&p)[3], const float* __restrict__ f, int nb, uint16_t* __restrict__ row)
{
	auto put = [&](int k, float v) {
		if (BF16) { const __nv_bfloat16 h = __float2bfloat16_rn(v); row[k] = *reinterpret_cast<const uint16_t*>(&h); }
		else { const __half h = __float2half_rn(v); row[k] = *reinterpret_cast<const uint16_t*>(&h); }
	};
#pragma unroll
	for (int c = 0; c < 3; c++) put(c, p[c]);
#pragma unroll 1
	for (int b = 0; b < nb; b++) {
		const float fb = f[b];
#pragma unroll
		for (int c = 0; c < 3; c++) {
			const float arg = __fmul_rn(p[c], fb);
			put(3 + 6 * b + c, sinf(arg));
			put(3 + 6 * b + 3 + c, cosf(arg));
		}
	}
}

template <bool TRAIN, bool RAW>
__global__ void __launch_bounds__(kThreads, 1) mlp_nerf_fwd_tc_kernel(const uint8_t* __restrict__ blob,
	const float* __restrict__ x, int64_t n, float* __restrict__ out, uint8_t* __restrict__ saved, const RawInput raw)
{
	extern __shared__ __align__(128) uint8_t smem_raw[];
	Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int64_t n_tiles = (n + 127) / 128;
	// every CTA runs the same number of rounds; a round past the last tile is a tile of no rows
	const int64_t my_tiles = (n_tiles + gridDim.x - 1) / gridDim.x;

	if (warp == 1) {
		if (lane == 0) {
			for (int s = 0; s < kRing; s++) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], 1); }
			mbar_init(&sm.a_ready, 4);
			mbar_init(&sm.d_ready, 1);
			asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		}
		__syncwarp();
		tmem_alloc_all(&sm.tmem_base);
	}
	for (int i = threadIdx.x; i < kBiasFloats; i += kThreads) sm.bias[i] = reinterpret_cast<const float*>(blob + kWeightBytes)[i];
	fence_before();
	__syncthreads();
	fence_after();
	const uint32_t tmem = sm.tmem_base;

	if (warp == 0) {
		// ===== producer: the same 41-stage weight stream for every tile =====
		if (lane == 0) {
			uint32_t g = 0;
			for (int64_t t = 0; t < my_tiles; t++) {
#pragma unroll 1
				for (int i = 0; i < kFwdStages; i++, g++) {
					const uint32_t slot = g % kRing, round = g / kRing;
					mbar_wait(&sm.empty[slot], (round & 1u) ^ 1u);          // first round passes immediately
					const uint32_t bytes = c_fwd_table.bytes[i];
					const int off = c_fwd_table.off[i];
					mbar_expect_tx(&sm.full[slot], bytes);
					tma_bulk_g2s(sm.ring[slot], blob + off, bytes, &sm.full[slot]);
				}
			}
		}
	} else if (warp == 1) {
		// ===== MMA issuer =====
		if (lane == 0) {
			uint32_t g = 0, pa = 0;
			for (int64_t t = 0; t < my_tiles; t++) {
#pragma unroll 1
				for (int grp = 0; grp < kGroups; grp++) {
					mbar_wait(&sm.a_ready, pa);
					pa ^= 1u;
					fence_after();
					for (int l = group_first(grp); l < group_first(grp) + group_count(grp); l++) {
						const LayerInfo L = layer_info(l);
						const uint32_t id = idesc(128, L.N, TRAIN, 0, 0);
						const uint32_t lbo = L.N * 16;
						uint32_t a_col = tmem + L.a_col;
						bool first = true;
						for (int s = 0; s < layer_stages(l); s++, g++) {
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
							umma_commit(&sm.empty[slot]);   // the stage is free again once these MMAs have read it
						}
					}
					umma_commit(&sm.d_ready);
				}
			}
		}
	} else {
		// ===== epilogue warps: one thread per row of the tile =====
		const int q = warp & 3;                                           // TMEM lane quarter this warp may access
		const int row = (q << 5) | lane;
		const uint32_t t_lane = tmem + (static_cast<uint32_t>(q << 5) << 16);
		uint32_t pd = 0;
		for (int64_t t = 0; t < my_tiles; t++) {
			const int64_t tile = blockIdx.x + t * gridDim.x;
			const int64_t r = tile * 128 + row;
			const bool ok = r < n;
			// rows past n of the last tile are stored too (finite; their gradients are zero); a round past the last tile stores into the
			// spare record that nrf_mlp_nerf_saved_bytes appends for this purpose
			uint8_t* const rec = TRAIN ? saved + (tile < n_tiles ? tile : n_tiles) * kSaveTile : nullptr;
			// ---- inputs: 63 point channels (+1 zero) and 27 view channels (+5 zero) as fp16 pairs into their TMEM columns
			if (RAW) {
				uint16_t* srow = sm.stage + row * kStagePitch;
				uint32_t* srow32 = reinterpret_cast<uint32_t*>(srow);
				if (ok) {
					float p[3], d[3];
					const int64_t ray = r / raw.samples_per_ray;
#pragma unroll
					for (int c = 0; c < 3; c++) { p[c] = __ldg(x + r * 3 + c); d[c] = __ldg(raw.dirs + ray * 3 + c); }
					posenc_stage<TRAIN>(p, raw.fp, 10, srow);
					srow[63] = 0;
					posenc_stage<TRAIN>(d, raw.fv, 4, srow + 64);
#pragma unroll
					for (int k = 27; k < 32; k++) srow[64 + k] = 0;
				} else {
#pragma unroll
					for (int i = 0; i < 48; i++) srow32[i] = 0u;
				}
				uint32_t a16[16];
#pragma unroll
				for (int h = 0; h < 2; h++) {
#pragma unroll
					for (int i = 0; i < 16; i++) a16[i] = srow32[16 * h + i];
					tmem_st16(t_lane + kColPts + 16 * h, a16);
					if (TRAIN) store_chunks(rec + kSavePts + chunk_offset(64, row, 0), 4 * h, a16);
				}
#pragma unroll
				for (int i = 0; i < 16; i++) a16[i] = srow32[32 + i];
				tmem_st16(t_lane + kColViews, a16);
				if (TRAIN) store_chunks(rec + kSaveViews + chunk_offset(32, row, 0), 0, a16);
			} else {
				const float2* xr = reinterpret_cast<const float2*>(x + (ok ? r : 0) * kInCh);   // rows are 360 B: 8-byte aligned
				uint32_t a16[16];
#pragma unroll
				for (int h = 0; h < 2; h++) {
#pragma unroll
					for (int i = 0; i < 16; i++) {
						const int k = 32 * h + 2 * i;
						float2 v = make_float2(0.f, 0.f);
						if (ok) {
							if (k + 1 < kInPts) v = __ldg(xr + k / 2);
							else if (k < kInPts) v = make_float2(__ldg(x + r * kInCh + k), 0.f);
						}
						a16[i] = TRAIN ? pack_bf16(v.x, v.y) : pack_f16(v.x, v.y);
					}
					tmem_st16(t_lane + kColPts + 16 * h, a16);
					if (TRAIN) store_chunks(rec + kSavePts + chunk_offset(64, row, 0), 4 * h, a16);
				}
#pragma unroll
				for (int i = 0; i < 16; i++) {
					const int k = 2 * i;
					float v0 = 0.f, v1 = 0.f;
					if (ok && k < kInViews) v0 = __ldg(x + r * kInCh + kInPts + k);
					if (ok && k + 1 < kInViews) v1 = __ldg(x + r * kInCh + kInPts + k + 1);
					a16[i] = TRAIN ? pack_bf16(v0, v1) : pack_f16(v0, v1);
				}
				tmem_st16(t_lane + kColViews, a16);
				if (TRAIN) store_chunks(rec + kSaveViews + chunk_offset(32, row, 0), 0, a16);
			}
			publish(&sm.a_ready, lane);

			float alpha = 0.f;
#pragma unroll 1
			for (int grp = 0; grp < kGroups; grp++) {
				mbar_wait(&sm.d_ready, pd);
				pd ^= 1u;
				fence_after();
				if (grp < 8) {
					// pts_linears: relu(D + b) -> h (the next layer's A operand)
					epilogue_to_h<8, true, TRAIN>(t_lane, sm.bias + bias_offset(0) + grp * kW, rec + save_h(grp + 1) + chunk_offset(256, row, 0), rec + bits_offset(grp + 1, row));
					publish(&sm.a_ready, lane);
				} else if (grp == 8) {
					// feature_linear (no activation) -> h ; alpha_linear -> register
					uint32_t d16[16];
					tmem_ld16(t_lane + kColD16, d16);
					tmem_ld_wait();
					alpha = __uint_as_float(d16[0]) + sm.bias[bias_offset(9)];
					epilogue_to_h<8, false, TRAIN>(t_lane, sm.bias + bias_offset(8), rec + kSaveFeat + chunk_offset(256, row, 0), nullptr);
					publish(&sm.a_ready, lane);
				} else if (grp == 9) {
					// views_linears[0]: relu -> first 128 channels of h
					epilogue_to_h<4, true, TRAIN>(t_lane, sm.bias + bias_offset(10), rec + kSaveHv + chunk_offset(128, row, 0), rec + bits_offset(0, row));
					publish(&sm.a_ready, lane);
				} else {
					// rgb_linear -> out = [rgb, alpha] (src/NeRF.cpp:119-120)
					uint32_t c4[4];
					tmem_ld4(t_lane + kColD16, c4);
					tmem_ld_wait();
					const float* b = sm.bias + bias_offset(11);
					if (ok) *reinterpret_cast<float4*>(out + r * 4) = make_float4(__uint_as_float(c4[0]) + b[0], __uint_as_float(c4[1]) + b[1],
						__uint_as_float(c4[2]) + b[2], alpha);
				}
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

int check_shape(const nrf_mlp_nerf_shape* s)
{
	NRF_REQUIRE(s != nullptr, "shape is null");
	if (!(s->depth == 8 && s->width == kW && s->input_ch == kInPts && s->input_ch_views == kInViews && s->skip_layer == 4 && s->use_viewdirs == 1)) {
		set_error("nrf_mlp_nerf: only the BASELINE shape D=8 W=256 in=63+27 skip={4} use_viewdirs is built");
		return NRF_ERR_UNSUPPORTED;
	}
	return NRF_OK;
}

}  // namespace nerf_tc
}  // namespace nrf

using namespace nrf;
using namespace nrf::nerf_tc;

template <bool TRAIN, bool RAW>
static int fwd_common(const nrf_mlp_nerf_shape* shape, const void* packed, const float* x, int64_t n, float* out, void* saved, const RawInput& raw,
	nrf_stream stream)
{
	if (int rc = nerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(n >= 0, "negative n");
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(packed && x && out && (!TRAIN || saved) && (!RAW || (raw.dirs && raw.samples_per_ray >= 1)), "null pointer");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 127) == 0 && (RAW || (reinterpret_cast<uintptr_t>(x) & 7) == 0) && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
		(reinterpret_cast<uintptr_t>(saved) & 127) == 0, "packed / saved must be 128-byte, x 8-byte, out 16-byte aligned");
	const int64_t tiles = (n + 127) / 128;
	const int smem = static_cast<int>(sizeof(Smem)) + 128;
	// Every CTA streams the whole weight blob for each of its tiles.  That L2 -> SM weight traffic does not pace this kernel: 2-CTA clusters
	// that shared one multicast weight stream halved it and measured equal (0.332 vs 0.330 ms at 196 608 rows).  What does: one tile in
	// flight, so a layer is its MMAs (16 x 128 cycles) THEN its epilogue, and the epilogue reads 128 KB of fp32 accumulators out of TMEM
	// at 64 B/clk (2 048 cycles) — splitting it over 8 warps instead of 4 gained 5 % (inference) / lost 7 % (training).
	const int blocks = static_cast<int>(std::min<int64_t>(tiles, kNumSMs));
	NRF_CUDA(cudaFuncSetAttribute(mlp_nerf_fwd_tc_kernel<TRAIN, RAW>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
	mlp_nerf_fwd_tc_kernel<TRAIN, RAW><<<blocks, kThreads, smem, as_stream(stream)>>>(reinterpret_cast<const uint8_t*>(packed), x, n, out,
		reinterpret_cast<uint8_t*>(saved), raw);
	NRF_CHECK_LAUNCH("mlp_nerf_fwd_tc_kernel");
	return NRF_OK;
}

static int make_raw(const float* dirs, int32_t samples_per_ray, const float* freqs_pts, int32_t n_freqs_pts, const float* freqs_views, int32_t n_freqs_views,
	RawInput& raw)
{
	NRF_REQUIRE(freqs_pts && freqs_views && n_freqs_pts == 10 && n_freqs_views == 4, "the fused embedding is built for multires 10 (points) and 4 (directions)");
	raw.dirs = dirs;
	raw.samples_per_ray = samples_per_ray;
	for (int i = 0; i < 10; i++) raw.fp[i] = freqs_pts[i];
	for (int i = 0; i < 4; i++) raw.fv[i] = freqs_views[i];
	return NRF_OK;
}

extern "C" {

int64_t nrf_mlp_nerf_packed_bytes(const nrf_mlp_nerf_shape* shape) { return nerf_tc::check_shape(shape) ? -1 : static_cast<int64_t>(kPackedBytes); }

static int pack_common(const nrf_mlp_nerf_shape* shape, const nrf_mlp_nerf_weights* w, void* packed, bool bf16, nrf_stream stream)
{
	if (int rc = nerf_tc::check_shape(shape)) return rc;
	NRF_REQUIRE(w != nullptr && packed != nullptr, "null pointer");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 127) == 0, "packed blob must be 128-byte aligned");
	Weights p;
	for (int i = 0; i < 8; i++) { p.w[i] = w->pts_w[i]; p.b[i] = w->pts_b[i]; }
	p.w[8] = w->feature_w; p.b[8] = w->feature_b;
	p.w[9] = w->alpha_w; p.b[9] = w->alpha_b;
	p.w[10] = w->views_w; p.b[10] = w->views_b;
	p.w[11] = w->rgb_w; p.b[11] = w->rgb_b;
	for (int i = 0; i < kLayers; i++) NRF_REQUIRE(p.w[i] && p.b[i], "null weight / bias pointer");
	nerf_pack_kernel<<<(kPackedBytes / 4 + 255) / 256, 256, 0, as_stream(stream)>>>(p, reinterpret_cast<uint32_t*>(packed), bf16);
	NRF_CHECK_LAUNCH("nerf_pack_kernel");
	return NRF_OK;
}

int nrf_mlp_nerf_pack(const nrf_mlp_nerf_shape* shape, const nrf_mlp_nerf_weights* w, void* packed, nrf_stream stream)
{
	return pack_common(shape, w, packed, false, stream);
}

int nrf_mlp_nerf_pack_train(const nrf_mlp_nerf_shape* shape, const nrf_mlp_nerf_weights* w, void* packed, nrf_stream stream)
{
	return pack_common(shape, w, packed, true, stream);
}

int64_t nrf_mlp_nerf_saved_bytes(const nrf_mlp_nerf_shape* shape, int64_t n)
{
	if (nerf_tc::check_shape(shape) || n < 0) return -1;
	return ((n + 127) / 128 + 1) * static_cast<int64_t>(kSaveTile);      // + one spare record (a CTA's rounds past the last tile write there)
}

int nrf_mlp_nerf_fwd(const nrf_mlp_nerf_shape* shape, const void* packed, const float* x, int64_t n, float* out, nrf_stream stream)
{
	return fwd_common<false, false>(shape, packed, x, n, out, nullptr, RawInput{}, stream);
}

int nrf_mlp_nerf_fwd_train(const nrf_mlp_nerf_shape* shape, const void* packed_train, const float* x, int64_t n, float* out, void* saved,
                           nrf_stream stream)
{
	return fwd_common<true, false>(shape, packed_train, x, n, out, saved, RawInput{}, stream);
}

int nrf_mlp_nerf_fwd_points(const nrf_mlp_nerf_shape* shape, const void* packed, const float* points, const float* dirs, int32_t samples_per_ray,
                            const float* freqs_pts_host, int32_t n_freqs_pts, const float* freqs_views_host, int32_t n_freqs_views, int64_t n, float* out,
                            nrf_stream stream)
{
	RawInput raw{};
	if (int rc = make_raw(dirs, samples_per_ray, freqs_pts_host, n_freqs_pts, freqs_views_host, n_freqs_views, raw)) return rc;
	return fwd_common<false, true>(shape, packed, points, n, out, nullptr, raw, stream);
}

int nrf_mlp_nerf_fwd_train_points(const nrf_mlp_nerf_shape* shape, const void* packed_train, const float* points, const float* dirs,
                                  int32_t samples_per_ray, const float* freqs_pts_host, int32_t n_freqs_pts, const float* freqs_views_host,
                                  int32_t n_freqs_views, int64_t n, float* out, void* saved, nrf_stream stream)
{
	RawInput raw{};
	if (int rc = make_raw(dirs, samples_per_ray, freqs_pts_host, n_freqs_pts, freqs_views_host, n_freqs_views, raw)) return rc;
	return fwd_common<true, true>(shape, packed_train, points, n, out, saved, raw, stream);
}

}
