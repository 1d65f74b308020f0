// Data-parallel optimiser step as ONE kernel over NVLink peer memory: reduce-scatter of the gradient + Adam on the owned
// shard + all-gather of the fp16 table shadow, fused (nrf_adam_step_sharded).
//
// The reference has no multi-GPU code; the plain data-parallel step is all-reduce(grad) [NCCL] -> dense Adam on every rank
// (nerfpp_b200/parallel.py).  Every rank then spends the full 48 us streaming ALL 8.9 M parameters and moments, and the
// all-reduce moves 2 (G-1)/G x 35.6 MB per GPU.  Here each rank OWNS a contiguous 1/G shard of the hash table:
//   phase 0   system-scope barrier: every peer's gradient is complete (flags in peer memory, monotone epochs);
//   phase 1   for the owned shard: g = sum over ranks (fixed rank order: bit-identical on every run) of the peers' gradient
//             slices, read straight from their HBM over NVLink (ld.global on mapped peer pointers); Adam on the local fp32
//             master / moments; the new value is rounded to fp16 and STORED INTO EVERY PEER'S SHADOW TABLE (st.global on
//             mapped peer pointers) — the forward pass only ever reads the fp16 shadow, so fp32 never crosses the link again;
//             the 9 344 MLP weights are not sharded: every rank reduces their gradients in the same order and keeps a replica;
//   phase 2   system-scope barrier: all shadows written, all gradients consumed; then the local gradient is cleared.
// Per GPU and step: (G-1)/G x 35.6 MB in, (G-1)/G x 17.8 MB out, Adam traffic / G.  Pointers come from
// torch.distributed._symmetric_memory (plumbing); the kernel itself is plain loads/stores on peer addresses.
#include "common.cuh"

namespace nrf {

struct AdamSchedState {   // optim.cu
	int32_t step;
	float lr_over_bc1, inv_sqrt_bc2, lr;
};

struct PeerArgs {
	int world, rank;
	const float* grads[NRF_MAX_PEERS];   // every rank's flat gradient (mapped peer memory; [rank] is local)
	__half* shadow[NRF_MAX_PEERS];       // every rank's fp16 parameter shadow
	uint32_t* flags[NRF_MAX_PEERS];      // every rank's flag block: [0,world) entry barrier, [world,2 world) exit barrier,
	                                     // [2 world] local epoch, [2 world + 1] local release word, [2 world + 2] timeout marker
	const float* grads_mc;               // multicast mapping of the gradient buffers (nullptr: none)
	__half* shadow_mc;                   // multicast mapping of the shadow buffers
};

// sum over all ranks of the 16 bytes at this multicast address, reduced in the NVSwitch
__device__ __forceinline__ float4 multimem_ld_reduce_add_v4(const float* mc)
{
	float4 v;
	asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
	return v;
}
__device__ __forceinline__ float multimem_ld_reduce_add(const float* mc)
{
	float v;
	asm volatile("multimem.ld_reduce.relaxed.sys.global.add.f32 %0, [%1];" : "=f"(v) : "l"(mc) : "memory");
	return v;
}
// the same 8 bytes into every rank's copy (the .f32 type only names the width: a store moves bits)
__device__ __forceinline__ void multimem_st_v2(void* mc, uint32_t a, uint32_t b)
{
	asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1,%2};" ::"l"(mc), "f"(__uint_as_float(a)), "f"(__uint_as_float(b)) : "memory");
}

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p)
{
	uint32_t v;
	asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
	return v;
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p)
{
	uint32_t v;
	asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
	return v;
}

// All CTAs of all ranks meet here.  CTA 0 / thread 0 raises this rank's slot in every peer's flag block to `epoch` and waits for
// every peer's slot in the local block; the other CTAs wait for the local release word.  Needs all CTAs co-resident (cooperative launch,
// grid <= SMs).  A rank that never arrives (crashed peer) releases the others after ~2 s: EVERY path that gives up sets the sticky
// timeout marker, and the barrier then returns false to the whole CTA — the caller must not write parameters, shadows or gradients after
// a failed barrier (the host reads the marker and raises: PeerShardedOptimizer.check).
__device__ __forceinline__ bool peer_barrier(const PeerArgs& a, int which, uint32_t epoch, uint32_t* done_counter)
{
	uint32_t* mine = a.flags[a.rank];
	uint32_t* marker = mine + 2 * a.world + 2;
	__shared__ int s_ok;
	__syncthreads();
	if (threadIdx.x == 0) {
		__threadfence_system();   // this CTA's peer stores / loads are ordered before its arrival
		const uint32_t target = 2u * (epoch - 1u) + which + 1u;       // value of the release word once this barrier has been passed (monotone over calls)
		const uint32_t arrived = atomicAdd(done_counter, 1u) + 1u;    // counts the arrivals of THIS call: reset at its end, so calls may differ in grid size
		if (arrived == gridDim.x * (which + 1u)) {
			// last CTA of this rank to arrive: tell the peers, wait for them, release the local CTAs
			for (int p = 0; p < a.world; p++) st_release_sys(a.flags[p] + which * a.world + a.rank, epoch);
			const long long t0 = clock64();
			bool late = false;
			for (int p = 0; p < a.world && !late; p++) {
				while (ld_acquire_sys(mine + which * a.world + p) < epoch) {
					if (clock64() - t0 > 4000000000LL) { late = true; break; }
				}
			}
			if (late) atomicExch(marker, 1u);
			st_release_sys(mine + 2 * a.world + 1, target);
		} else {
			const long long t0 = clock64();
			while (ld_acquire_gpu(mine + 2 * a.world + 1) < target) {
				if (clock64() - t0 > 6000000000LL) { atomicExch(marker, 1u); break; }
			}
		}
		__threadfence_system();
		s_ok = ld_acquire_gpu(marker) == 0u;
	}
	__syncthreads();
	return s_ok != 0;
}

__device__ __forceinline__ uint32_t globaltimer_lo()
{
	uint32_t t;
	asm volatile("mov.u32 %0, %%globaltimer_lo;" : "=r"(t));
	return t;
}
// phase timestamps (ns, low word) of CTA 0 in words [kStampBase, kStampBase + 5) of the local flag block: kernel entry, after the
// entry barrier, after the shard loop, after the exit barrier, after the gradient clear — read back by scripts/exp/dp_step.py
constexpr int kStampBase = 2 * NRF_MAX_PEERS + 8;

__device__ __forceinline__ float adam_update(float p, float g, float& m, float& v, float beta1, float beta2, float eps, float lr_over_bc1,
	float inv_sqrt_bc2)
{
	m = m * beta1 + g * (1.f - beta1);
	v = v * beta2 + g * g * (1.f - beta2);
	const float denom = sqrtf(v) * inv_sqrt_bc2 + eps;
	return p - lr_over_bc1 * (m / denom);
}

// n_sharded: leading scalars partitioned over the ranks in contiguous shards (multiple of 4 per shard boundary);
// [n_sharded, n_total): replicated tail (every rank reduces and updates it identically).
// WORLD is a template parameter so that the peer loop unrolls and all W x U remote 16-byte loads of an iteration are in flight
// together (NVLink round trips are ~2 us: the kernel lives on memory-level parallelism).
// MC: the gradient sum of a quad is ONE multimem.ld_reduce on the multicast mapping and the fp16 result ONE multimem.st, instead of WORLD peer
// loads and WORLD peer stores: per GPU and step 1/W x 35.6 MB arrives reduced (4.5 MB at W = 8) instead of (W-1)/W x 35.6 MB.
// The kernel takes its two regions as ranges: the sharded scalars [range_lo, range_hi) (multiples of 4; partitioned over the ranks) and the
// replicated scalars [tail_lo, tail_hi).  nrf_adam_step_sharded launches it over the whole flat vector: [0, n_sharded / 4 * 4) and the rest.
template <int WORLD, int U, bool MC>
__global__ void __launch_bounds__(512, 1) adam_sharded_kernel(PeerArgs a, float* __restrict__ param, float* __restrict__ m, float* __restrict__ v,
	float* grad_local, int64_t range_lo, int64_t range_hi, int64_t tail_lo, int64_t tail_hi, const AdamSchedState* __restrict__ sched, float beta1,
	float beta2, float eps, float grad_scale)
{
	uint32_t* mine = a.flags[a.rank];
	__shared__ uint32_t s_epoch, s_dead;
	if (threadIdx.x == 0) {
		s_epoch = mine[2 * WORLD] + 1u;   // every CTA reads the epoch before anyone bumps it (bumped after barrier 1)
		s_dead = mine[2 * WORLD + 2];     // sticky: an earlier step lost a peer -> this and every later step write nothing
	}
	__syncthreads();
	if (s_dead) return;
	const uint32_t epoch = s_epoch;
	uint32_t* done_counter = mine + 2 * WORLD + 3;
	const bool stamp = blockIdx.x == 0 && threadIdx.x == 0;
	if (stamp) mine[kStampBase + 0] = globaltimer_lo();

	if (!peer_barrier(a, 0, epoch, done_counter)) return;   // some peer's gradient may be incomplete: touch nothing
	if (stamp) mine[kStampBase + 1] = globaltimer_lo();

	const float lr_over_bc1 = sched->lr_over_bc1, inv_sqrt_bc2 = sched->inv_sqrt_bc2;
	// shard bounds in units of 4 scalars
	const int64_t quads = (range_hi - range_lo) / 4;
	const int64_t base = quads / WORLD, extra = quads % WORLD;
	const int64_t q_lo = range_lo / 4 + a.rank * base + (a.rank < extra ? a.rank : extra);
	const int64_t q_hi = q_lo + base + (a.rank < extra ? 1 : 0);
	const int64_t tid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	const int64_t nthreads = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t q0 = q_lo + tid; q0 < q_hi; q0 += nthreads * U) {
		float4 g4[U][WORLD], p4[U], m4[U], v4[U];
#pragma unroll
		for (int u = 0; u < U; u++) {
			const int64_t q = q0 + u * nthreads;
			if (q < q_hi) {
				if (MC) {
					g4[u][0] = multimem_ld_reduce_add_v4(a.grads_mc + q * 4);
				} else {
#pragma unroll
					for (int p = 0; p < WORLD; p++) g4[u][p] = *reinterpret_cast<const float4*>(a.grads[p] + q * 4);
				}
				p4[u] = *reinterpret_cast<float4*>(param + q * 4);
				m4[u] = *reinterpret_cast<float4*>(m + q * 4);
				v4[u] = *reinterpret_cast<float4*>(v + q * 4);
			}
		}
#pragma unroll
		for (int u = 0; u < U; u++) {
			const int64_t q = q0 + u * nthreads;
			if (q >= q_hi) continue;
			const int64_t i = q * 4;
			float4 g = g4[u][0];
			if (!MC) {
#pragma unroll
				for (int p = 1; p < WORLD; p++) { g.x += g4[u][p].x; g.y += g4[u][p].y; g.z += g4[u][p].z; g.w += g4[u][p].w; }   // fixed rank order
			}
			float4 pp = p4[u], mm = m4[u], vv = v4[u];
			pp.x = adam_update(pp.x, g.x * grad_scale, mm.x, vv.x, beta1, beta2, eps, lr_over_bc1, inv_sqrt_bc2);
			pp.y = adam_update(pp.y, g.y * grad_scale, mm.y, vv.y, beta1, beta2, eps, lr_over_bc1, inv_sqrt_bc2);
			pp.z = adam_update(pp.z, g.z * grad_scale, mm.z, vv.z, beta1, beta2, eps, lr_over_bc1, inv_sqrt_bc2);
			pp.w = adam_update(pp.w, g.w * grad_scale, mm.w, vv.w, beta1, beta2, eps, lr_over_bc1, inv_sqrt_bc2);
			*reinterpret_cast<float4*>(param + i) = pp;
			*reinterpret_cast<float4*>(m + i) = mm;
			*reinterpret_cast<float4*>(v + i) = vv;
			__half2 lo = __floats2half2_rn(pp.x, pp.y), hi = __floats2half2_rn(pp.z, pp.w);
			uint2 o;
			o.x = *reinterpret_cast<uint32_t*>(&lo);
			o.y = *reinterpret_cast<uint32_t*>(&hi);
			if (MC) {
				multimem_st_v2(a.shadow_mc + i, o.x, o.y);                                     // all-gather of the fp16 shadow through the switch
			} else {
#pragma unroll
				for (int p = 0; p < WORLD; p++) *reinterpret_cast<uint2*>(a.shadow[p] + i) = o;   // all-gather of the fp16 shadow
			}
		}
	}
	// the replicated scalars (the MLP weights, and what of the table does not fill a quad): every rank, same order
	for (int64_t i = tail_lo + tid; i < tail_hi; i += nthreads) {
		float g = 0.f;
		if (MC) {
			g = multimem_ld_reduce_add(a.grads_mc + i);       // every rank reads the same switch-reduced sum: the replicas of the tail stay identical
		} else {
#pragma unroll
			for (int p = 0; p < WORLD; p++) g += a.grads[p][i];
		}
		float mm = m[i], vv = v[i];
		const float pn = adam_update(param[i], g * grad_scale, mm, vv, beta1, beta2, eps, lr_over_bc1, inv_sqrt_bc2);
		param[i] = pn; m[i] = mm; v[i] = vv;
		a.shadow[a.rank][i] = __float2half_rn(pn);
	}

	if (stamp) mine[kStampBase + 2] = globaltimer_lo();
	if (!peer_barrier(a, 1, epoch, done_counter)) return;   // a peer may still be reading this rank's gradient: do not clear it
	if (stamp) mine[kStampBase + 3] = globaltimer_lo();

	// every peer has consumed this call's part of this rank's gradient: clear it for the next step
	for (int64_t q = range_lo / 4 + tid; q < range_hi / 4; q += nthreads) *reinterpret_cast<float4*>(grad_local + q * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
	for (int64_t i = tail_lo + tid; i < tail_hi; i += nthreads) grad_local[i] = 0.f;
	if (tid == 0) {
		mine[2 * WORLD] = epoch;
		*done_counter = 0u;   // every CTA of this call has arrived at both barriers (the exit barrier was released): the next call counts from zero
	}
	if (stamp) mine[kStampBase + 4] = globaltimer_lo();
}

}  // namespace nrf

using namespace nrf;

extern "C" {

int64_t nrf_peer_flags_bytes(int32_t world) { return world >= 1 && world <= NRF_MAX_PEERS ? (kStampBase + 8) * 4 : -1; }

int nrf_adam_step_sharded(const nrf_peer_group* pg, float* param, float* exp_avg, float* exp_avg_sq, int64_t n_sharded, int64_t n_total,
	const void* sched_state, float beta1, float beta2, float eps, float grad_scale, nrf_stream stream)
{
	NRF_REQUIRE(n_sharded >= 0 && n_total >= n_sharded, "bad sizes");
	NRF_REQUIRE(pg != nullptr && pg->world >= 1 && pg->world <= NRF_MAX_PEERS && pg->rank >= 0 && pg->rank < pg->world, "bad peer group");
	if (n_total == 0) return NRF_OK;
	const int64_t q4 = n_sharded / 4 * 4;   // sharded: whole quads of the table; replicated: [q4, n_total)
	NRF_REQUIRE(param && exp_avg && exp_avg_sq && sched_state, "null pointer");
	PeerArgs a;
	a.world = pg->world; a.rank = pg->rank;
	for (int p = 0; p < pg->world; p++) {
		NRF_REQUIRE(pg->grads[p] && pg->shadow_f16[p] && pg->flags[p], "null peer pointer");
		NRF_REQUIRE(((reinterpret_cast<uintptr_t>(pg->grads[p]) & 15) | (reinterpret_cast<uintptr_t>(pg->shadow_f16[p]) & 7)) == 0, "peer buffers must be 16-byte aligned");
		a.grads[p] = pg->grads[p];
		a.shadow[p] = reinterpret_cast<__half*>(pg->shadow_f16[p]);
		a.flags[p] = pg->flags[p];
	}
	NRF_REQUIRE(((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(exp_avg) | reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0,
		"buffers must be 16-byte aligned");
	// one CTA per SM, all co-resident: the in-kernel barriers need every CTA of the grid running
	int sms = kNumSMs;
	int dev = 0;
	if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
	// cooperative launch: the driver guarantees that all CTAs are co-resident (or refuses the launch) — the in-kernel barriers spin
	float* grad_local = const_cast<float*>(a.grads[a.rank]);
	const AdamSchedState* sched = reinterpret_cast<const AdamSchedState*>(sched_state);
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = dim3(sms);
	cfg.blockDim = dim3(512);
	cfg.dynamicSmemBytes = 0;
	cfg.stream = as_stream(stream);
	cudaLaunchAttribute attr[1];
	attr[0].id = cudaLaunchAttributeCooperative;
	attr[0].val.cooperative = 1;
	cfg.attrs = attr;
	cfg.numAttrs = 1;
	cudaError_t launch_err = cudaSuccess;
	a.grads_mc = pg->grads_mc;
	a.shadow_mc = reinterpret_cast<__half*>(pg->shadow_f16_mc);
	const bool mc = pg->grads_mc != nullptr && pg->shadow_f16_mc != nullptr && pg->world > 1;
	NRF_REQUIRE(!mc || (((reinterpret_cast<uintptr_t>(pg->grads_mc) & 15) | (reinterpret_cast<uintptr_t>(pg->shadow_f16_mc) & 7)) == 0), "multicast mappings must be 16-byte aligned");
#define NRF_LAUNCH_SHARDED(W, U)                                                                                                                 \
	launch_err = mc ? cudaLaunchKernelEx(&cfg, adam_sharded_kernel<W, 4, true>, a, param, exp_avg, exp_avg_sq, grad_local, 0, q4, q4, n_total,  \
	                      sched, beta1, beta2, eps, grad_scale)                                                                                  \
	                : cudaLaunchKernelEx(&cfg, adam_sharded_kernel<W, U, false>, a, param, exp_avg, exp_avg_sq, grad_local, 0, q4, q4, n_total, \
	                      sched, beta1, beta2, eps, grad_scale)
	switch (pg->world) {
		case 1: NRF_LAUNCH_SHARDED(1, 4); break;
		case 2: NRF_LAUNCH_SHARDED(2, 4); break;
		case 3: NRF_LAUNCH_SHARDED(3, 2); break;
		case 4: NRF_LAUNCH_SHARDED(4, 2); break;
		case 5: NRF_LAUNCH_SHARDED(5, 2); break;
		case 6: NRF_LAUNCH_SHARDED(6, 2); break;
		case 7: NRF_LAUNCH_SHARDED(7, 2); break;
		default: NRF_LAUNCH_SHARDED(8, 2); break;
	}
#undef NRF_LAUNCH_SHARDED
	if (launch_err != cudaSuccess) { set_error("adam_sharded_kernel: %s", cudaGetErrorString(launch_err)); cudaGetLastError(); return NRF_ERR_CUDA; }
	NRF_CHECK_LAUNCH("adam_sharded_kernel");
	return NRF_OK;
}

}
