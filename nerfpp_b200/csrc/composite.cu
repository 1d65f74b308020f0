// Per-ray alpha compositing (forward and backward) for sm_100a.
//
// Replaces NeRFRenderer::RawToOutputs (reference src/NeRFRenderer.h:199-282) — about 25 ATen launches that
// each stream an [R,S] temporary — and folds TruncExp (src/CustomOps.cpp:5-16) in.  One launch each way:
//   * one warp per ray, lane = sample inside a 32-sample block, so raw (float4 per sample), z and the weights
//     are read / written as fully coalesced 512 B / 128 B warp transactions;
//   * the transmittance is the reference's log-space form: an exclusive prefix SUM of log(max(1-alpha,1e-10))
//     done with warp shuffles plus a running carry across blocks, then TruncExp;
//   * the backward recomputes the forward from raw (nothing saved) and turns the cumsum adjoint into a
//     reverse (suffix) warp scan.
// HBM traffic: 24 B/sample + 44 B/ray forward, 24 B in + 16 B out per sample backward (SURVEY §8d).
#include "common.cuh"

namespace nrf {

constexpr int kRaysPerCta = 8;       // warps

struct SampleEval {
	float r, g, b;     // sigmoid(rgb logits)
	float alpha, x;    // alpha = 1 - exp(x), x = -relu(sigma)*dist
	float dist, sig;   // interval length * |d|, density after noise
	float ell;         // log(max(1-alpha, 1e-10))
};

__device__ __forceinline__ float sigmoidf_(float v) { return 1.f / (1.f + expf(-v)); }

__device__ __forceinline__ float ray_norm(const float* __restrict__ rays_d, int64_t ray)
{
	const float dx = rays_d[ray * 3], dy = rays_d[ray * 3 + 1], dz = rays_d[ray * 3 + 2];
	return sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
}

// the global-memory operands of one sample: loaded for every block of a ray BEFORE any arithmetic (composite_fwd_nb_kernel,
// composite_bwd_kernel), so a warp has all its sectors in flight at once instead of one 32-sample block per memory round trip
struct SampleIn {
	float4 v;          // raw[..., 0:4]
	float zi, zn;      // z[i], z[i+1]
	float noise;
};

__device__ __forceinline__ SampleIn load_sample(const float* __restrict__ raw, int raw_stride, const float* __restrict__ zrow,
	const float* __restrict__ noise_row, int i, int S)
{
	SampleIn in;
	if (raw_stride == 4) in.v = *reinterpret_cast<const float4*>(raw + static_cast<int64_t>(i) * 4);
	else {
		const float* p = raw + static_cast<int64_t>(i) * raw_stride;
		in.v = make_float4(p[0], p[1], p[2], p[3]);
	}
	in.zi = zrow[i];
	in.zn = (i + 1 < S) ? zrow[i + 1] : 0.f;
	in.noise = noise_row ? noise_row[i] : 0.f;
	return in;
}

// src/NeRFRenderer.h:239-256 for one sample
__device__ __forceinline__ SampleEval eval_loaded(const SampleIn& in, bool has_noise, float noise_std, float dnorm, int i, int S)
{
	SampleEval e;
	const float4 v = in.v;
	e.r = sigmoidf_(v.x);
	e.g = sigmoidf_(v.y);
	e.b = sigmoidf_(v.z);
	const float d = (i + 1 < S) ? __fsub_rn(in.zn, in.zi) : 1e10f;
	e.dist = __fmul_rn(d, dnorm);
	float sig = v.w;
	if (has_noise) sig = __fadd_rn(sig, __fmul_rn(in.noise, noise_std));
	e.sig = sig;
	e.x = -__fmul_rn(fmaxf(sig, 0.f), e.dist);
	// S == 1 reproduces a reference quirk: `dists` is built from z[...,1:]-z[...,:-1] ([R,0]) and the 1e10 tail is
	// expanded to that EMPTY shape (src/NeRFRenderer.h:239-240), so every [R,S] tensor is empty and all maps are zero.
	e.alpha = (S == 1) ? 0.f : 1.f - expf(e.x);
	e.ell = logf(fmaxf(1.f - e.alpha, 1e-10f));
	return e;
}

__device__ __forceinline__ SampleEval eval_sample(const float* __restrict__ raw, int raw_stride, const float* __restrict__ zrow,
	const float* __restrict__ noise_row, float noise_std, float dnorm, int i, int S)
{
	return eval_loaded(load_sample(raw, raw_stride, zrow, noise_row, i, S), noise_row != nullptr, noise_std, dnorm, i, S);
}

__global__ void __launch_bounds__(kRaysPerCta * 32) composite_fwd_kernel(const float* __restrict__ raw, int raw_stride,
	const float* __restrict__ z, const float* __restrict__ rays_d, const float* __restrict__ noise, float noise_std, int white,
	int64_t R, int S, float* __restrict__ rgb, float* __restrict__ depth, float* __restrict__ disp, float* __restrict__ acc,
	float* __restrict__ weights)
{
	const int lane = threadIdx.x & 31;
	const int64_t ray = static_cast<int64_t>(blockIdx.x) * kRaysPerCta + (threadIdx.x >> 5);
	if (ray >= R) return;
	const float* raw_row = raw + ray * S * raw_stride;
	const float* zrow = z + ray * S;
	const float* nrow = (noise && noise_std > 0.f) ? noise + ray * S : nullptr;
	const float dnorm = ray_norm(rays_d, ray);

	float carry = 0.f, sr = 0.f, sg = 0.f, sb = 0.f, sa = 0.f, sd = 0.f;
	for (int b0 = 0; b0 < S; b0 += 32) {
		const int i = b0 + lane;
		float ell = 0.f, w = 0.f;
		SampleEval e;
		if (i < S) {
			e = eval_sample(raw_row, raw_stride, zrow, nrow, noise_std, dnorm, i, S);
			ell = e.ell;
		}
		const float incl = warp_scan_incl(ell, lane);
		const float T = expf(carry + (incl - ell));  // TruncExp forward is a plain exp (src/CustomOps.cpp:8)
		if (i < S) {
			w = e.alpha * T;
			sr += w * e.r;
			sg += w * e.g;
			sb += w * e.b;
			sa += w;
			sd += w * zrow[i];
			if (weights) weights[ray * S + i] = w;
		}
		carry += __shfl_sync(0xffffffffu, incl, 31);
	}
	sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb); sa = warp_sum(sa); sd = warp_sum(sd);
	if (lane == 0) {
		if (white) {
			const float bg = 1.f - sa;
			sr += bg; sg += bg; sb += bg;
		}
		if (rgb) { rgb[ray * 3] = sr; rgb[ray * 3 + 1] = sg; rgb[ray * 3 + 2] = sb; }
		const float dep = sd / fmaxf(sa, 1e-10f);
		if (depth) depth[ray] = dep;
		if (disp) disp[ray] = 1.f / fmaxf(1e-10f, dep);
		if (acc) acc[ray] = sa;
	}
}

// S <= 32 * NB: the same arithmetic with every load of the ray issued up front
template <int NB>
__global__ void __launch_bounds__(kRaysPerCta * 32) composite_fwd_nb_kernel(const float* __restrict__ raw, int raw_stride,
	const float* __restrict__ z, const float* __restrict__ rays_d, const float* __restrict__ noise, float noise_std, int white,
	int64_t R, int S, float* __restrict__ rgb, float* __restrict__ depth, float* __restrict__ disp, float* __restrict__ acc,
	float* __restrict__ weights)
{
	const int lane = threadIdx.x & 31;
	const int64_t ray = static_cast<int64_t>(blockIdx.x) * kRaysPerCta + (threadIdx.x >> 5);
	if (ray >= R) return;
	const float* raw_row = raw + ray * S * raw_stride;
	const float* zrow = z + ray * S;
	const float* nrow = (noise && noise_std > 0.f) ? noise + ray * S : nullptr;
	SampleIn in[NB];
#pragma unroll
	for (int b = 0; b < NB; b++) {
		const int i = b * 32 + lane;
		if (i < S) in[b] = load_sample(raw_row, raw_stride, zrow, nrow, i, S);
	}
	const float dnorm = ray_norm(rays_d, ray);

	float carry = 0.f, sr = 0.f, sg = 0.f, sb = 0.f, sa = 0.f, sd = 0.f;
#pragma unroll
	for (int b = 0; b < NB; b++) {
		const int i = b * 32 + lane;
		float ell = 0.f, w = 0.f;
		SampleEval e;
		if (i < S) {
			e = eval_loaded(in[b], nrow != nullptr, noise_std, dnorm, i, S);
			ell = e.ell;
		}
		const float incl = warp_scan_incl(ell, lane);
		const float T = expf(carry + (incl - ell));  // TruncExp forward is a plain exp (src/CustomOps.cpp:8)
		if (i < S) {
			w = e.alpha * T;
			sr += w * e.r;
			sg += w * e.g;
			sb += w * e.b;
			sa += w;
			sd += w * in[b].zi;
			if (weights) weights[ray * S + i] = w;
		}
		carry += __shfl_sync(0xffffffffu, incl, 31);
	}
	sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb); sa = warp_sum(sa); sd = warp_sum(sd);
	if (lane == 0) {
		if (white) {
			const float bg = 1.f - sa;
			sr += bg; sg += bg; sb += bg;
		}
		if (rgb) { rgb[ray * 3] = sr; rgb[ray * 3 + 1] = sg; rgb[ray * 3 + 2] = sb; }
		const float dep = sd / fmaxf(sa, 1e-10f);
		if (depth) depth[ray] = dep;
		if (disp) disp[ray] = 1.f / fmaxf(1e-10f, dep);
		if (acc) acc[ray] = sa;
	}
}

// The training tail of the colour pass as ONE kernel (HUBER): RawToOutputs forward of the ray (recomputed here anyway), the huber loss of its
// RGB against the target (src/NeRFExecutor.h:883-886: mean over all R*3 values, delta 1) and the backward — instead of composite forward ->
// huber -> composite backward with an [R,3] gradient round trip and two more launches.
struct HuberArgs {
	const float* target;     // [R,3]
	float delta, grad_scale;
	float inv_n;             // 1 / (R * 3)
	float* loss_out;         // += mean loss
	float* rgb_out;          // [R,3] nullable
};

template <int NB, bool HUBER>
__global__ void __launch_bounds__(kRaysPerCta * 32) composite_bwd_kernel(const float* __restrict__ raw, int raw_stride,
	const float* __restrict__ z, const float* __restrict__ rays_d, const float* __restrict__ noise, float noise_std, int white,
	int64_t R, int S, const float* __restrict__ g_rgb, const float* __restrict__ g_depth, const float* __restrict__ g_disp,
	const float* __restrict__ g_acc, const float* __restrict__ g_weights, float* __restrict__ d_raw, HuberArgs hub)
{
	const int lane = threadIdx.x & 31;
	const int64_t ray = static_cast<int64_t>(blockIdx.x) * kRaysPerCta + (threadIdx.x >> 5);
	if (ray >= R) return;
	const float* raw_row = raw + ray * S * raw_stride;
	const float* zrow = z + ray * S;
	const float* nrow = (noise && noise_std > 0.f) ? noise + ray * S : nullptr;
	const float dnorm = ray_norm(rays_d, ray);

	SampleEval e[NB];
	float Lx[NB];  // exclusive log-transmittance
	float zi[NB];
	float carry = 0.f, sa = 0.f, sd = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
	{
		SampleIn in[NB];
#pragma unroll
		for (int b = 0; b < NB; b++) {
			const int i = b * 32 + lane;
			if (i < S) in[b] = load_sample(raw_row, raw_stride, zrow, nrow, i, S);
		}
#pragma unroll
		for (int b = 0; b < NB; b++) {
			const int i = b * 32 + lane;
			zi[b] = i < S ? in[b].zi : 0.f;
			e[b] = i < S ? eval_loaded(in[b], nrow != nullptr, noise_std, dnorm, i, S) : SampleEval{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
		}
	}
#pragma unroll
	for (int b = 0; b < NB; b++) {
		const int i = b * 32 + lane;
		float ell = 0.f;
		if (i < S) {
			ell = e[b].ell;
		}
		const float incl = warp_scan_incl(ell, lane);
		Lx[b] = carry + (incl - ell);
		if (i < S) {
			const float w = e[b].alpha * expf(Lx[b]);
			sa += w;
			sd += w * zi[b];
			if (HUBER) { sr += w * e[b].r; sg += w * e[b].g; sb += w * e[b].b; }
		}
		carry += __shfl_sync(0xffffffffu, incl, 31);
	}
	sa = warp_sum(sa);
	sd = warp_sum(sd);

	float gr, gg, gb;
	if (HUBER) {
		// the forward's RGB of this ray (same sums as composite_fwd_nb_kernel), then d huber / d rgb
		sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
		if (white) { const float bg = 1.f - sa; sr += bg; sg += bg; sb += bg; }
		const float er = sr - hub.target[ray * 3], eg = sg - hub.target[ray * 3 + 1], eb = sb - hub.target[ray * 3 + 2];
		const float d = hub.delta;
		gr = (fabsf(er) < d ? er : (er > 0.f ? d : -d)) * hub.inv_n * hub.grad_scale;      // the expression of huber_kernel (optim.cu)
		gg = (fabsf(eg) < d ? eg : (eg > 0.f ? d : -d)) * hub.inv_n * hub.grad_scale;
		gb = (fabsf(eb) < d ? eb : (eb > 0.f ? d : -d)) * hub.inv_n * hub.grad_scale;
		if (lane == 0) {
			const float l = (fabsf(er) < d ? 0.5f * er * er : d * (fabsf(er) - 0.5f * d)) + (fabsf(eg) < d ? 0.5f * eg * eg : d * (fabsf(eg) - 0.5f * d)) +
			                (fabsf(eb) < d ? 0.5f * eb * eb : d * (fabsf(eb) - 0.5f * d));
			if (hub.loss_out) atomicAdd(hub.loss_out, l * hub.inv_n);
			if (hub.rgb_out) { hub.rgb_out[ray * 3] = sr; hub.rgb_out[ray * 3 + 1] = sg; hub.rgb_out[ray * 3 + 2] = sb; }
		}
	} else {
		gr = g_rgb ? g_rgb[ray * 3] : 0.f; gg = g_rgb ? g_rgb[ray * 3 + 1] : 0.f; gb = g_rgb ? g_rgb[ray * 3 + 2] : 0.f;
	}
	const float den = fmaxf(sa, 1e-10f);
	const float dep = sd / den;
	float gdep = g_depth ? g_depth[ray] : 0.f;
	if (g_disp && dep > 1e-10f) gdep += g_disp[ray] * (-1.f / (dep * dep));  // disp = 1/max(1e-10, depth)
	float gacc = g_acc ? g_acc[ray] : 0.f;
	if (white) gacc -= (gr + gg + gb);                                     // rgb += 1 - acc
	if (sa >= 1e-10f) gacc -= gdep * sd / (den * den);                     // clamp_min passes the gradient
	const float gz = gdep / den;

	float rcarry = 0.f;  // sum of dL over samples after the current block
#pragma unroll
	for (int b = NB - 1; b >= 0; b--) {
		const int i = b * 32 + lane;
		const bool ok = i < S;
		float G = 0.f, T = 0.f, dL = 0.f;
		if (ok) {
			T = expf(Lx[b]);
			G = gr * e[b].r + gg * e[b].g + gb * e[b].b + gacc + gz * zi[b];
			if (g_weights) G += g_weights[ray * S + i];
			dL = G * e[b].alpha * expf(fminf(fmaxf(Lx[b], -100.f), 5.f));  // TruncExp backward (src/CustomOps.cpp:14)
		}
		const float incl = warp_scan_incl_rev(dL, lane);
		const float dell = rcarry + (incl - dL);  // sum over samples strictly after i
		rcarry += __shfl_sync(0xffffffffu, incl, 0);
		if (ok) {
			float dalpha = G * T;
			const float om = 1.f - e[b].alpha;
			if (om >= 1e-10f) dalpha -= dell / om;
			const float dx = -dalpha * expf(fminf(fmaxf(e[b].x, -100.f), 5.f));
			const float dsig = (e[b].sig > 0.f && S > 1) ? -e[b].dist * dx : 0.f;
			const float w = e[b].alpha * T;
			float4 o;
			o.x = w * gr * e[b].r * (1.f - e[b].r);
			o.y = w * gg * e[b].g * (1.f - e[b].g);
			o.z = w * gb * e[b].b * (1.f - e[b].b);
			o.w = dsig;
			*reinterpret_cast<float4*>(d_raw + (ray * S + i) * 4) = o;
		}
	}
}

// Any S (the kernels above keep a ray's S <= 256 samples in registers): two passes over the ray in 32-sample blocks.  Pass 1 re-evaluates the
// forward (sums, and the log-transmittance carried into every block, kept in shared memory); pass 2 walks the blocks backwards, evaluating each
// sample again, with the suffix sum of dL carried across blocks.  Same expressions, same order of the scans as composite_bwd_kernel.
constexpr int kGenericMaxBlocks = 64;   // S <= 2048

template <bool HUBER>
__global__ void __launch_bounds__(kRaysPerCta * 32) composite_bwd_generic_kernel(const float* __restrict__ raw, int raw_stride,
	const float* __restrict__ z, const float* __restrict__ rays_d, const float* __restrict__ noise, float noise_std, int white,
	int64_t R, int S, const float* __restrict__ g_rgb, const float* __restrict__ g_depth, const float* __restrict__ g_disp,
	const float* __restrict__ g_acc, const float* __restrict__ g_weights, float* __restrict__ d_raw, HuberArgs hub)
{
	__shared__ float block_carry[kRaysPerCta][kGenericMaxBlocks];
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	const int64_t ray = static_cast<int64_t>(blockIdx.x) * kRaysPerCta + wid;
	if (ray >= R) return;
	const float* raw_row = raw + ray * S * raw_stride;
	const float* zrow = z + ray * S;
	const float* nrow = (noise && noise_std > 0.f) ? noise + ray * S : nullptr;
	const float dnorm = ray_norm(rays_d, ray);
	const int nb = (S + 31) / 32;
	const SampleEval none{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};

	float carry = 0.f, sa = 0.f, sd = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
	for (int b = 0; b < nb; b++) {
		const int i = b * 32 + lane;
		SampleEval e = none;
		float zi = 0.f;
		if (i < S) {
			const SampleIn in = load_sample(raw_row, raw_stride, zrow, nrow, i, S);
			zi = in.zi;
			e = eval_loaded(in, nrow != nullptr, noise_std, dnorm, i, S);
		}
		const float ell = i < S ? e.ell : 0.f;
		const float incl = warp_scan_incl(ell, lane);
		if (lane == 0) block_carry[wid][b] = carry;
		if (i < S) {
			const float w = e.alpha * expf(carry + (incl - ell));
			sa += w;
			sd += w * zi;
			if (HUBER) { sr += w * e.r; sg += w * e.g; sb += w * e.b; }
		}
		carry += __shfl_sync(0xffffffffu, incl, 31);
	}
	__syncwarp();
	sa = warp_sum(sa);
	sd = warp_sum(sd);
	float gr, gg, gb;
	if (HUBER) {
		sr = warp_sum(sr); sg = warp_sum(sg); sb = warp_sum(sb);
		if (white) { const float bg = 1.f - sa; sr += bg; sg += bg; sb += bg; }
		const float er = sr - hub.target[ray * 3], eg = sg - hub.target[ray * 3 + 1], eb = sb - hub.target[ray * 3 + 2];
		const float d = hub.delta;
		gr = (fabsf(er) < d ? er : (er > 0.f ? d : -d)) * hub.inv_n * hub.grad_scale;
		gg = (fabsf(eg) < d ? eg : (eg > 0.f ? d : -d)) * hub.inv_n * hub.grad_scale;
		gb = (fabsf(eb) < d ? eb : (eb > 0.f ? d : -d)) * hub.inv_n * hub.grad_scale;
		if (lane == 0) {
			const float l = (fabsf(er) < d ? 0.5f * er * er : d * (fabsf(er) - 0.5f * d)) + (fabsf(eg) < d ? 0.5f * eg * eg : d * (fabsf(eg) - 0.5f * d)) +
			                (fabsf(eb) < d ? 0.5f * eb * eb : d * (fabsf(eb) - 0.5f * d));
			if (hub.loss_out) atomicAdd(hub.loss_out, l * hub.inv_n);
			if (hub.rgb_out) { hub.rgb_out[ray * 3] = sr; hub.rgb_out[ray * 3 + 1] = sg; hub.rgb_out[ray * 3 + 2] = sb; }
		}
	} else {
		gr = g_rgb ? g_rgb[ray * 3] : 0.f; gg = g_rgb ? g_rgb[ray * 3 + 1] : 0.f; gb = g_rgb ? g_rgb[ray * 3 + 2] : 0.f;
	}
	const float den = fmaxf(sa, 1e-10f);
	const float dep = sd / den;
	float gdep = g_depth ? g_depth[ray] : 0.f;
	if (g_disp && dep > 1e-10f) gdep += g_disp[ray] * (-1.f / (dep * dep));
	float gacc = g_acc ? g_acc[ray] : 0.f;
	if (white) gacc -= (gr + gg + gb);
	if (sa >= 1e-10f) gacc -= gdep * sd / (den * den);
	const float gz = gdep / den;

	float rcarry = 0.f;
	for (int b = nb - 1; b >= 0; b--) {
		const int i = b * 32 + lane;
		const bool ok = i < S;
		SampleEval e = none;
		float zi = 0.f;
		if (ok) {
			const SampleIn in = load_sample(raw_row, raw_stride, zrow, nrow, i, S);
			zi = in.zi;
			e = eval_loaded(in, nrow != nullptr, noise_std, dnorm, i, S);
		}
		const float ell = ok ? e.ell : 0.f;
		const float Lx = block_carry[wid][b] + (warp_scan_incl(ell, lane) - ell);
		float G = 0.f, T = 0.f, dL = 0.f;
		if (ok) {
			T = expf(Lx);
			G = gr * e.r + gg * e.g + gb * e.b + gacc + gz * zi;
			if (g_weights) G += g_weights[ray * S + i];
			dL = G * e.alpha * expf(fminf(fmaxf(Lx, -100.f), 5.f));
		}
		const float incl = warp_scan_incl_rev(dL, lane);
		const float dell = rcarry + (incl - dL);
		rcarry += __shfl_sync(0xffffffffu, incl, 0);
		if (ok) {
			float dalpha = G * T;
			const float om = 1.f - e.alpha;
			if (om >= 1e-10f) dalpha -= dell / om;
			const float dx = -dalpha * expf(fminf(fmaxf(e.x, -100.f), 5.f));
			const float dsig = (e.sig > 0.f && S > 1) ? -e.dist * dx : 0.f;
			const float w = e.alpha * T;
			float4 o;
			o.x = w * gr * e.r * (1.f - e.r);
			o.y = w * gg * e.g * (1.f - e.g);
			o.z = w * gb * e.b * (1.f - e.b);
			o.w = dsig;
			*reinterpret_cast<float4*>(d_raw + (ray * S + i) * 4) = o;
		}
	}
}

}  // namespace nrf

using namespace nrf;

extern "C" {

int nrf_composite_fwd(const float* raw, int32_t raw_stride, const float* z, const float* rays_d, const float* noise,
	float raw_noise_std, int32_t white_bkgr, int64_t n_rays, int32_t n_samples, float* rgb, float* depth, float* disp,
	float* acc, float* weights, nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1, "bad sizes");
	NRF_REQUIRE(raw_stride >= 4, "raw_stride must be >= 4");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(raw && z && rays_d, "null input");
	const unsigned blocks = static_cast<unsigned>((n_rays + kRaysPerCta - 1) / kRaysPerCta);
	cudaStream_t s = as_stream(stream);
	const int nb = (n_samples + 31) / 32;
#define NRF_CF(NBV)                                                                                                     \
	case NBV:                                                                                                           \
		composite_fwd_nb_kernel<NBV><<<blocks, kRaysPerCta * 32, 0, s>>>(raw, raw_stride, z, rays_d, noise, raw_noise_std, \
			white_bkgr, n_rays, n_samples, rgb, depth, disp, acc, weights);                                              \
		break
	switch (nb) {
		NRF_CF(1); NRF_CF(2); NRF_CF(3); NRF_CF(4); NRF_CF(5); NRF_CF(6); NRF_CF(7); NRF_CF(8);
		default:
			composite_fwd_kernel<<<blocks, kRaysPerCta * 32, 0, s>>>(raw, raw_stride, z, rays_d, noise, raw_noise_std, white_bkgr, n_rays,
				n_samples, rgb, depth, disp, acc, weights);
	}
#undef NRF_CF
	NRF_CHECK_LAUNCH("composite_fwd_kernel");
	return NRF_OK;
}

int nrf_composite_bwd(const float* raw, int32_t raw_stride, const float* z, const float* rays_d, const float* noise,
	float raw_noise_std, int32_t white_bkgr, int64_t n_rays, int32_t n_samples, const float* g_rgb, const float* g_depth,
	const float* g_disp, const float* g_acc, const float* g_weights, float* d_raw, nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1, "bad sizes");
	NRF_REQUIRE(raw_stride >= 4, "raw_stride must be >= 4");
	NRF_REQUIRE(n_samples <= 32 * kGenericMaxBlocks, "n_samples > 2048 is not supported by the backward");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(raw && z && rays_d && d_raw, "null input");
	const unsigned blocks = static_cast<unsigned>((n_rays + kRaysPerCta - 1) / kRaysPerCta);
	cudaStream_t s = as_stream(stream);
	const int nb = (n_samples + 31) / 32;
	const HuberArgs none{};
#define NRF_CB(NBV)                                                                                                  \
	case NBV:                                                                                                        \
		composite_bwd_kernel<NBV, false><<<blocks, kRaysPerCta * 32, 0, s>>>(raw, raw_stride, z, rays_d, noise, raw_noise_std, \
			white_bkgr, n_rays, n_samples, g_rgb, g_depth, g_disp, g_acc, g_weights, d_raw, none);                    \
		break
	switch (nb) {
		NRF_CB(1); NRF_CB(2); NRF_CB(3); NRF_CB(4); NRF_CB(5); NRF_CB(6); NRF_CB(7); NRF_CB(8);
		default:   // more samples than a warp keeps in registers: the two-pass kernel
			composite_bwd_generic_kernel<false><<<blocks, kRaysPerCta * 32, 0, s>>>(raw, raw_stride, z, rays_d, noise, raw_noise_std, white_bkgr, n_rays,
				n_samples, g_rgb, g_depth, g_disp, g_acc, g_weights, d_raw, none);
	}
#undef NRF_CB
	NRF_CHECK_LAUNCH("composite_bwd_kernel");
	return NRF_OK;
}

int nrf_composite_huber_bwd(const float* raw, int32_t raw_stride, const float* z, const float* rays_d, const float* noise, float raw_noise_std,
	int32_t white_bkgr, int64_t n_rays, int32_t n_samples, const float* target, float delta, float grad_scale, float* loss_out, float* rgb_out,
	float* d_raw, nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1, "bad sizes");
	NRF_REQUIRE(raw_stride >= 4, "raw_stride must be >= 4");
	NRF_REQUIRE(n_samples <= 32 * kGenericMaxBlocks, "n_samples > 2048 is not supported by the backward");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(raw && z && rays_d && d_raw && target, "null input");
	const unsigned blocks = static_cast<unsigned>((n_rays + kRaysPerCta - 1) / kRaysPerCta);
	cudaStream_t s = as_stream(stream);
	const int nb = (n_samples + 31) / 32;
	HuberArgs hub;
	hub.target = target; hub.delta = delta; hub.inv_n = 1.f / static_cast<float>(n_rays * 3); hub.grad_scale = grad_scale;
	hub.loss_out = loss_out; hub.rgb_out = rgb_out;
#define NRF_CH(NBV)                                                                                                  \
	case NBV:                                                                                                        \
		composite_bwd_kernel<NBV, true><<<blocks, kRaysPerCta * 32, 0, s>>>(raw, raw_stride, z, rays_d, noise, raw_noise_std, \
			white_bkgr, n_rays, n_samples, static_cast<const float*>(nullptr), static_cast<const float*>(nullptr), static_cast<const float*>(nullptr), \
			static_cast<const float*>(nullptr), static_cast<const float*>(nullptr), d_raw, hub);                      \
		break
	switch (nb) {
		NRF_CH(1); NRF_CH(2); NRF_CH(3); NRF_CH(4); NRF_CH(5); NRF_CH(6); NRF_CH(7); NRF_CH(8);
		default:
			composite_bwd_generic_kernel<true><<<blocks, kRaysPerCta * 32, 0, s>>>(raw, raw_stride, z, rays_d, noise, raw_noise_std, white_bkgr, n_rays,
				n_samples, nullptr, nullptr, nullptr, nullptr, nullptr, d_raw, hub);
	}
#undef NRF_CH
	NRF_CHECK_LAUNCH("composite_bwd_kernel");
	return NRF_OK;
}

}
