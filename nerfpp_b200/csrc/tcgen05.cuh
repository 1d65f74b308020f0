// tcgen05 / TMEM / TMA / mbarrier PTX wrappers and the operand formats shared by the tensor-core kernels (NeRFSmall: mlp_small.cu,
// mlp_small_tc.cu; classic NeRF: mlp_nerf_tc.cu, mlp_nerf_bwd_tc.cu; LeRF head: lerf_tc.cu, lerf_bwd_tc.cu), sm_100a only: descriptor
// bits, the K-major core-matrix order of packed weights, the training-record chunking and the TMEM store -> fence -> arrive hand-off.
#pragma once
#include "common.cuh"

namespace nrf {
namespace tc {

// ---- PTX wrappers --------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity)
{
	uint32_t ok;
	asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
	             : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
	return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
	asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
	             ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// TMA 1-D bulk copy global -> shared, completion counted on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
	             ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// asynchronous L2 prefetch of a contiguous global range (bytes: multiple of 16)
__device__ __forceinline__ void tma_prefetch_l2(const void* src, uint32_t bytes)
{
	asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
// true in exactly one lane of a converged warp (the pattern the compiler recognises for single-thread tcgen05 issue)
__device__ __forceinline__ bool elect_one()
{
	uint32_t pred;
	asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
	return pred != 0;
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc_all(uint32_t* dst_smem)
{
	asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(dst_smem)) : "memory");
	asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free_all(uint32_t base)
{
	asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(base) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T, one K=16 step
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
	asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
	             ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, one K=16 step
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
	asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
	             ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
	asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// KSTEPS K = 16 steps of one accumulator block with the A operand in TMEM and an MN-major B operand: A advances 8 TMEM columns, the B
// descriptor 256 bytes (16 rows of K) per step; the first step accumulates onto D iff acc_first
template <int KSTEPS>
__device__ __forceinline__ void issue_k(uint32_t d, uint32_t a0, uint64_t b0, uint32_t idesc, uint32_t acc_first)
{
#pragma unroll
	for (int j = 0; j < KSTEPS; j++) umma_ts(d, a0 + 8 * j, b0 + static_cast<uint64_t>(16 * j), idesc, j ? 1u : acc_first);
}

// tcgen05.ld / st, shape 32x32b: thread i of the warp owns TMEM lane (32*(warp%4) + i) and gets / gives consecutive columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32])
{
	asm volatile(
		"tcgen05.ld.sync.aligned.32x32b.x32.b32 "
		"{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
		: "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
		  "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
		  "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
		  "=r"(r[31])
		: "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16])
{
	asm volatile(
		"tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
		: "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
		  "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
		: "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&r)[4])
{
	asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// the same wait, tied to the destination registers of an earlier tcgen05.ld so that no use of them can be scheduled above it
// (needed when another tcgen05.ld is issued between the load and its wait)
__device__ __forceinline__ void tmem_ld_wait_for(uint32_t (&r)[32])
{
	asm volatile("tcgen05.wait::ld.sync.aligned;"
		: "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]),
		  "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]),
		  "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]),
		  "+r"(r[31])
		:: "memory");
}
__device__ __forceinline__ void tmem_ld_wait_for(uint32_t (&r)[16])
{
	asm volatile("tcgen05.wait::ld.sync.aligned;"
		: "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]),
		  "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
		:: "memory");
}
__device__ __forceinline__ void tmem_ld_wait_for(uint32_t (&r)[4])
{
	asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]) :: "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16])
{
	asm volatile(
		"tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
		::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
		  "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
		: "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8])
{
	asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
		::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
// hand the A operand this warp just wrote to TMEM to the issuing thread: wait for the stores, fence, one mbarrier arrival per warp
__device__ __forceinline__ void publish(uint64_t* bar, int lane)
{
	tmem_st_wait();
	fence_before();
	__syncwarp();
	if (lane == 0) mbar_arrive(bar);
}

// ---- 16-bit pairs --------------------------------------------------------------------------------------------------
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

// ---- descriptors ---------------------------------------------------------------------------------------------------
// instruction descriptor, kind::f16: D fp32 (bits 4-5 = 1), A and B both fp16 (bf16 = false: bits 7-9, 10-12 = 0) or both bf16 (= 1),
// majors 0 = K, 1 = MN (bits 15, 16), N>>3 at bit 17, M>>4 at bit 24 (cute::UMMA::InstrDescriptor)
__host__ __device__ constexpr uint32_t idesc(int M, int N, bool bf16, int a_mn, int b_mn)
{
	return (1u << 4) | (bf16 ? (1u << 7) | (1u << 10) : 0u) | (uint32_t(a_mn) << 15) | (uint32_t(b_mn) << 16) | (uint32_t(N >> 3) << 17) |
	       (uint32_t(M >> 4) << 24);
}
// the shapes in use: forwards (fp16 K x K; classic-NeRF training bf16), gradient chains (bf16 K x MN), weight gradients (bf16 MN x MN)
static_assert(idesc(128, 64, false, 0, 0) == 0x08100010u && idesc(128, 16, false, 0, 0) == 0x08040010u &&
              idesc(128, 256, false, 0, 0) == 0x08400010u && idesc(128, 48, false, 0, 0) == 0x080c0010u, "fp16, K x K");
static_assert(idesc(128, 256, true, 0, 0) == 0x08400490u && idesc(128, 16, true, 0, 0) == 0x08040490u, "bf16, K x K");
static_assert(idesc(128, 128, true, 0, 1) == 0x08210490u && idesc(128, 32, true, 0, 1) == 0x08090490u, "bf16, K x MN");
static_assert(idesc(128, 64, true, 1, 1) == 0x08118490u && idesc(128, 80, true, 1, 1) == 0x08158490u &&
              idesc(128, 16, true, 1, 1) == 0x08058490u, "bf16, MN x MN");
// shared-memory matrix descriptor, no swizzle, K-major: start>>4 | LBO>>4 <<16 | SBO>>4 <<32 | version 1 <<46
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
	return uint64_t((saddr & 0x3FFFF) >> 4) | (uint64_t(lbo_bytes >> 4) << 16) | (uint64_t(sbo_bytes >> 4) << 32) | (uint64_t(1) << 46);
}

// ---- packed weights: K-major core matrices -------------------------------------------------------------------------
// A stage of N rows (outputs) holds element (n, k) at byte (k/8)*(N*16) + n*16 + (k%8)*2: 8 x 16-byte core matrices, SBO 128 B between
// 8-row groups and LBO N*16 B between K chunks.  Word q of the stage holds (n, k) and (n, k + 1); k_off is the stage's first column.
struct StageWord {
	int n, k;
};
__host__ __device__ __forceinline__ StageWord stage_word(int q, int N, int k_off)
{
	const int kc = q / (4 * N);
	return {(q >> 2) % N, k_off + 8 * kc + 2 * (q & 3)};
}

// ---- training records ----------------------------------------------------------------------------------------------
// Regions of C columns stored as [row half (2)][C/8 column chunks][64 rows][8 elements] of 16 bits per 128-row tile: a 64-row half of a
// region is at the same time the MN-major A operand (M = columns, K = rows) and the MN-major B operand (N = columns, K = rows) of a
// weight-gradient product dW = dY^T X (SBO 1024, LBO 128).
__host__ __device__ constexpr int region_bytes(int cols) { return 128 * cols * 2; }
// byte offset of the 16-byte chunk (row r, columns 8*chunk ..) inside a region of `cols` columns
__host__ __device__ constexpr uint32_t chunk_offset(int cols, int r, int chunk)
{
	return static_cast<uint32_t>((r >> 6) * (cols * 128) + chunk * 1024 + (r & 63) * 16);
}
// 32 packed columns (16 words) of this thread's row -> chunks first_chunk .. first_chunk + 3 of a region (region_row: the row's chunk 0)
__device__ __forceinline__ void store_chunks(uint8_t* __restrict__ region_row, int first_chunk, const uint32_t (&a16)[16])
{
#pragma unroll
	for (int i = 0; i < 4; i++)
		*reinterpret_cast<uint4*>(region_row + (first_chunk + i) * 1024) = make_uint4(a16[4 * i], a16[4 * i + 1], a16[4 * i + 2], a16[4 * i + 3]);
}

}  // namespace tc
}  // namespace nrf
