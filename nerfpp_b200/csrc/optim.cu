// Loss and optimiser kernels restated from the training lines of NeRFExecutor::Train
// (reference src/NeRFExecutor.h:883-890 huber_loss(delta=1, mean); :539 Adam(betas 0.9/0.99, eps 1e-15); :986 step()).
//
// The Adam kernel is one streaming pass over param/grad/m/v (28 B read + 12..18 B written per scalar) that also
//   * clears the gradient for the next step (no separate 34..64 MiB memset), and
//   * refreshes the fp16 shadow of the hash table, which removes the reference's per-forward full-table
//     fp32->fp16 cast (src/CuHashEmbedder.cu:257: 96 MiB of traffic per forward call).
#include "common.cuh"

namespace nrf {

__global__ void __launch_bounds__(256) huber_kernel(const float* __restrict__ pred, const float* __restrict__ target, int64_t n,
	float delta, float grad_scale, float inv_n, float* __restrict__ loss_out, float* __restrict__ grad)
{
	float part = 0.f;
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		const float e = pred[i] - target[i];
		const float ae = fabsf(e);
		part += ae < delta ? 0.5f * e * e : delta * (ae - 0.5f * delta);
		if (grad) grad[i] = (ae < delta ? e : (e > 0.f ? delta : -delta)) * inv_n * grad_scale;
	}
	part = warp_sum(part);
	__shared__ float red[8];
	if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
	__syncthreads();
	if (threadIdx.x < 8) {
		float v = red[threadIdx.x];
#pragma unroll
		for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(0xffu, v, o);
		if (threadIdx.x == 0 && loss_out) atomicAdd(loss_out, v * inv_n);
	}
}

struct AdamArgs {
	float lr_over_bc1;   // lr / (1 - beta1^t)
	float inv_sqrt_bc2;  // 1 / sqrt(1 - beta2^t)
	float beta1, beta2, eps, grad_scale;
};

__device__ __forceinline__ float adam_one(float p, float g, float& m, float& v, const AdamArgs& a)
{
	// torch/csrc/api/src/optim/adam.cpp: exp_avg.mul_(b1).add_(g, 1-b1); exp_avg_sq.mul_(b2).addcmul_(g, g, 1-b2);
	// denom = exp_avg_sq.sqrt() / sqrt(bias_correction2) + eps; p.addcdiv_(exp_avg, denom, -lr / bias_correction1)
	m = m * a.beta1 + g * (1.f - a.beta1);
	v = v * a.beta2 + g * g * (1.f - a.beta2);
	const float denom = sqrtf(v) * a.inv_sqrt_bc2 + a.eps;
	return p - a.lr_over_bc1 * (m / denom);
}

// Device-resident schedule (nrf_adam_schedule_advance): lets a captured CUDA graph replay the optimiser with a step count,
// bias corrections and decayed learning rate that advance on the device.
struct AdamSchedState {
	int32_t step;         // completed optimiser steps
	float lr_over_bc1;    // lr / (1 - beta1^step)
	float inv_sqrt_bc2;   // 1 / sqrt(1 - beta2^step)
	float lr;             // decayed rate used by this step
};

__global__ void adam_schedule_kernel(AdamSchedState* st, double lr0, double decay_rate, double decay_steps, double beta1, double beta2)
{
	if (threadIdx.x != 0 || blockIdx.x != 0) return;
	const int step = st->step + 1;
	// src/NeRFExecutor.h:986-996: step() runs with the rate set at the END of the previous iteration, lr0 * rate^(global_step / decay_steps)
	// with global_step counted from 0 and incremented after the update  =>  exponent (step - 2) / decay_steps, clamped at 0
	const int e = step - 2 > 0 ? step - 2 : 0;
	const double lr = decay_steps > 0.0 ? lr0 * pow(decay_rate, static_cast<double>(e) / decay_steps) : lr0;
	const double bc1 = 1.0 - pow(beta1, static_cast<double>(step));
	const double bc2 = 1.0 - pow(beta2, static_cast<double>(step));
	st->step = step;
	st->lr = static_cast<float>(lr);
	st->lr_over_bc1 = static_cast<float>(lr / bc1);
	st->inv_sqrt_bc2 = static_cast<float>(1.0 / sqrt(bc2));
}

// L2 residency hints.  The step streams 303 MB through the 126 MB L2 here; without hints the two arrays the NEXT step reads at random —
// the fp16 shadow (17.8 MB: hash encode gathers) and the zeroed gradient (35.6 MB: hash backward REDs) — are evicted by the fp32
// master / moment streams and the next coarse-pass encode starts cold.  Masters and moments are marked evict_first, shadow and gradient
// zeros evict_last.  A/B against plain loads and stores on the same B200, 100 graph-replayed steps each: adam_step 51.3 -> 46.4 us,
// step 0.8683 -> 0.8613 ms (profiles/r1_adam_l2hint_ab.json).
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
	uint64_t p;
	asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
	return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last()
{
	uint64_t p;
	asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
	return p;
}
__device__ __forceinline__ float4 ld_hint(const float* p, uint64_t pol)
{
	float4 v;
	asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
	return v;
}
__device__ __forceinline__ void st_hint(float* p, const float4& v, uint64_t pol)
{
	asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_hint2(void* p, uint32_t a, uint32_t b, uint64_t pol)
{
	asm volatile("st.global.L2::cache_hint.v2.b32 [%0], {%1, %2}, %3;" ::"l"(p), "r"(a), "r"(b), "l"(pol) : "memory");
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ param, float* __restrict__ grad, float* __restrict__ m,
	float* __restrict__ v, int64_t n, AdamArgs a, int zero_grad, __half* __restrict__ shadow, const AdamSchedState* __restrict__ sched)
{
	if (sched) {
		a.lr_over_bc1 = sched->lr_over_bc1;
		a.inv_sqrt_bc2 = sched->inv_sqrt_bc2;
	}
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x * 4;
	const uint64_t pol_first = l2_policy_evict_first(), pol_last = l2_policy_evict_last();
	for (int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
		if (i + 3 < n) {
			float4 p4 = ld_hint(param + i, pol_first), m4 = ld_hint(m + i, pol_first), v4 = ld_hint(v + i, pol_first);
			float4 g4 = *reinterpret_cast<float4*>(grad + i);
			p4.x = adam_one(p4.x, g4.x * a.grad_scale, m4.x, v4.x, a);
			p4.y = adam_one(p4.y, g4.y * a.grad_scale, m4.y, v4.y, a);
			p4.z = adam_one(p4.z, g4.z * a.grad_scale, m4.z, v4.z, a);
			p4.w = adam_one(p4.w, g4.w * a.grad_scale, m4.w, v4.w, a);
			const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
			__half2 lo = __floats2half2_rn(p4.x, p4.y), hi = __floats2half2_rn(p4.z, p4.w);
			st_hint(param + i, p4, pol_first);
			st_hint(m + i, m4, pol_first);
			st_hint(v + i, v4, pol_first);
			if (zero_grad) st_hint(grad + i, zero, pol_last);
			if (shadow) st_hint2(shadow + i, *reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi), pol_last);
		} else {
			for (int64_t j = i; j < n; j++) {
				float mm = m[j], vv = v[j];
				const float p = adam_one(param[j], grad[j] * a.grad_scale, mm, vv, a);
				param[j] = p; m[j] = mm; v[j] = vv;
				if (zero_grad) grad[j] = 0.f;
				if (shadow) shadow[j] = __float2half_rn(p);
			}
		}
	}
}

}  // namespace nrf

using namespace nrf;

extern "C" {

int nrf_huber_fwd_bwd(const float* pred, const float* target, int64_t n, float delta, float grad_scale, float* loss_out,
	float* grad, nrf_stream stream)
{
	NRF_REQUIRE(n >= 0, "bad size");
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(pred && target, "null pointer");
	const int blocks = static_cast<int>(std::min<int64_t>((n + 255) / 256, kNumSMs * 4));
	huber_kernel<<<blocks, 256, 0, as_stream(stream)>>>(pred, target, n, delta, grad_scale, 1.f / static_cast<float>(n), loss_out, grad);
	NRF_CHECK_LAUNCH("huber_kernel");
	return NRF_OK;
}

int nrf_adam_step(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
	float eps, int32_t step, float grad_scale, int32_t zero_grad, void* shadow_f16, nrf_stream stream)
{
	NRF_REQUIRE(n >= 0 && step >= 1, "bad size / step");
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(param && grad && exp_avg && exp_avg_sq, "null pointer");
	NRF_REQUIRE(((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(grad) | reinterpret_cast<uintptr_t>(exp_avg) |
	              reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0, "buffers must be 16-byte aligned");
	NRF_REQUIRE(!shadow_f16 || (reinterpret_cast<uintptr_t>(shadow_f16) & 7) == 0, "shadow must be 8-byte aligned");
	AdamArgs a;
	const double bc1 = 1.0 - std::pow(static_cast<double>(beta1), step);
	const double bc2 = 1.0 - std::pow(static_cast<double>(beta2), step);
	a.lr_over_bc1 = static_cast<float>(lr / bc1);
	a.inv_sqrt_bc2 = static_cast<float>(1.0 / std::sqrt(bc2));
	a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.grad_scale = grad_scale;
	const int64_t quads = (n + 3) / 4;
	const int blocks = static_cast<int>(std::min<int64_t>((quads + 255) / 256, kNumSMs * 8));
	adam_kernel<<<blocks, 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, a, zero_grad, reinterpret_cast<__half*>(shadow_f16), nullptr);
	NRF_CHECK_LAUNCH("adam_kernel");
	return NRF_OK;
}

int nrf_adam_schedule_advance(void* sched_state, float lr0, float decay_rate, float decay_steps, float beta1, float beta2, nrf_stream stream)
{
	NRF_REQUIRE(sched_state != nullptr, "null schedule state");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(sched_state) & 15) == 0, "schedule state must be 16-byte aligned");
	adam_schedule_kernel<<<1, 32, 0, as_stream(stream)>>>(reinterpret_cast<AdamSchedState*>(sched_state), static_cast<double>(lr0),
		static_cast<double>(decay_rate), static_cast<double>(decay_steps), static_cast<double>(beta1), static_cast<double>(beta2));
	NRF_CHECK_LAUNCH("adam_schedule_kernel");
	return NRF_OK;
}

int nrf_adam_step_scheduled(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const void* sched_state, float beta1,
	float beta2, float eps, float grad_scale, int32_t zero_grad, void* shadow_f16, nrf_stream stream)
{
	NRF_REQUIRE(n >= 0, "bad size");
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(param && grad && exp_avg && exp_avg_sq && sched_state, "null pointer");
	NRF_REQUIRE(((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(grad) | reinterpret_cast<uintptr_t>(exp_avg) |
	              reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0, "buffers must be 16-byte aligned");
	NRF_REQUIRE(!shadow_f16 || (reinterpret_cast<uintptr_t>(shadow_f16) & 7) == 0, "shadow must be 8-byte aligned");
	AdamArgs a;
	a.lr_over_bc1 = 0.f; a.inv_sqrt_bc2 = 0.f;   // taken from sched_state on the device
	a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.grad_scale = grad_scale;
	const int64_t quads = (n + 3) / 4;
	const int blocks = static_cast<int>(std::min<int64_t>((quads + 255) / 256, kNumSMs * 8));
	adam_kernel<<<blocks, 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, a, zero_grad,
		reinterpret_cast<__half*>(shadow_f16), reinterpret_cast<const AdamSchedState*>(sched_state));
	NRF_CHECK_LAUNCH("adam_kernel");
	return NRF_OK;
}

}
