// Inverse-CDF importance sampling (+ merge with the coarse samples) for sm_100a.
//
// Replaces SamplePDF (reference src/Sampler.h:6-43: ~20 ATen launches, gathers through expanded
// [R,N,63] views, an H2D copy of `u` per call) and the torch::sort of cat(z, z_samples) at
// src/NeRFRenderer.h:427-431.  One warp per ray:
//   pdf/cdf  : weights+1e-8, sum by warp reduction, cdf = [0, cumsum(pdf)] by warp prefix scan (shared memory);
//   invert   : searchsorted(cdf, u, right=true) as a branch-free binary search per sample, then the
//              reference's below/above gather, `denom < 1e-5 -> 1` guard and lerp;
//   merge    : both lists are sorted when u is, so the sort is a rank merge (two binary searches per element);
//              for per-ray random u the S+N values are sorted with an in-warp bitonic network instead.
// Traffic: (2S + N + S+N) floats per ray, about 1.3 KB/ray at S=64, N=128 (SURVEY §8d).
#include "common.cuh"

namespace nrf {

constexpr int kSamplerWarps = 4;

// number of entries of the ascending array a[0..n) that are <= v  (searchsorted right=true).  Branch-free descent over power-of-two steps:
// the trip count depends on n only (warp-uniform), each step is one predicated load and a select — about half the instructions of the
// lo / hi loop, and the kernels here are bound by instruction issue.
__device__ __forceinline__ int upper_bound(const float* a, int n, float v)
{
	int pos = 0;
	for (int step = 1 << (31 - __clz(n | 1)); step > 0; step >>= 1) {
		const int p = pos + step;
		if (p <= n && a[p - 1] <= v) pos = p;
	}
	return pos;
}

// number of entries that are < v
__device__ __forceinline__ int lower_bound(const float* a, int n, float v)
{
	int pos = 0;
	for (int step = 1 << (31 - __clz(n | 1)); step > 0; step >>= 1) {
		const int p = pos + step;
		if (p <= n && a[p - 1] < v) pos = p;
	}
	return pos;
}

// inclusive prefix sum / max across the warp
__device__ __forceinline__ double warp_scan_incl_f64(double v, int lane)
{
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) {
		const double n = __shfl_up_sync(0xffffffffu, v, o);
		if (lane >= o) v += n;
	}
	return v;
}
__device__ __forceinline__ float warp_scan_max(float v, int lane)
{
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) {
		const float n = __shfl_up_sync(0xffffffffu, v, o);
		if (lane >= o) v = fmaxf(v, n);
	}
	return v;
}

// cdf[0..B) from weights[0..B-1) — src/Sampler.h:10-13.  All lanes of the warp call this.
// Summation order of sum()/cumsum() is implementation-defined in LibTorch (CPU cumsum accumulates in double,
// at::acc_type<float,false>; the CUDA one is a blocked fp32 scan).  Here both run in fp64 and are rounded to fp32
// once, i.e. each cdf knot is the correctly rounded prefix sum: equal to the CPU result and order independent.
// A prefix max then makes the knots monotone by construction, which the binary search and the rank merge rely on.
__device__ __forceinline__ void build_cdf(const float* __restrict__ w, int nw, float* cdf, int lane)
{
	double part = 0.0;
	for (int k = lane; k < nw; k += 32) part += static_cast<double>(__fadd_rn(w[k], 1e-8f));
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
	const float total = static_cast<float>(part);
	double carry = 0.0;
	float carry_max = 0.f;
	if (lane == 0) cdf[0] = 0.f;
	for (int k0 = 0; k0 < nw; k0 += 32) {
		const int k = k0 + lane;
		const float pdf = k < nw ? __fdiv_rn(__fadd_rn(w[k], 1e-8f), total) : 0.f;
		const double incl = warp_scan_incl_f64(static_cast<double>(pdf), lane);
		const float knot = fmaxf(warp_scan_max(static_cast<float>(carry + incl), lane), carry_max);
		if (k < nw) cdf[k + 1] = knot;
		carry += __shfl_sync(0xffffffffu, incl, 31);
		carry_max = __shfl_sync(0xffffffffu, knot, 31);
	}
	__syncwarp();
}

// src/Sampler.h:28-40 for one u
__device__ __forceinline__ float invert_cdf(const float* cdf, const float* bins, int B, float u)
{
	const int inds = upper_bound(cdf, B, u);
	const int below = max(0, inds - 1);
	const int above = min(B - 1, inds);
	const float c0 = cdf[below], c1 = cdf[above];
	const float b0 = bins[below], b1 = bins[above];
	float denom = __fsub_rn(c1, c0);
	if (denom < 1e-5f) denom = 1.f;
	const float t = __fdiv_rn(__fsub_rn(u, c0), denom);
	return __fadd_rn(b0, __fmul_rn(t, __fsub_rn(b1, b0)));
}

__device__ __forceinline__ void bitonic_sort(float* a, int n_pow2, int lane)
{
	for (int k = 2; k <= n_pow2; k <<= 1) {
		for (int j = k >> 1; j > 0; j >>= 1) {
			for (int i = lane; i < n_pow2; i += 32) {
				const int p = i ^ j;
				if (p > i) {
					const float x = a[i], y = a[p];
					const bool up = (i & k) == 0;
					if ((x > y) == up) { a[i] = y; a[p] = x; }
				}
			}
			__syncwarp();
		}
	}
}

// a[0..n) in shared memory, sorted except for rounding-level inversions -> sorted (odd-even transposition, whole warp)
__device__ __forceinline__ void restore_order(float* a, int n, int lane)
{
	for (;;) {
		bool swapped = false;
#pragma unroll
		for (int phase = 0; phase < 2; phase++) {
			for (int j = 2 * lane + phase; j + 1 < n; j += 64) {
				const float x = a[j], y = a[j + 1];
				if (x > y) { a[j] = y; a[j + 1] = x; swapped = true; }
			}
			__syncwarp();
		}
		if (!__any_sync(0xffffffffu, swapped)) break;
	}
}

// shared memory per warp: cdf[B] bins[B] zs[N] zc[S] (+ sort scratch when u is per-ray)
__global__ void __launch_bounds__(kSamplerWarps * 32) sample_pdf_merge_kernel(const float* __restrict__ z_coarse,
	const float* __restrict__ weights, const float* __restrict__ u, int u_per_ray, int64_t R, int S, int N,
	float* __restrict__ z_samples, float* __restrict__ z_merged, int16_t* __restrict__ perm_out, const float4* __restrict__ rows_coarse,
	float4* __restrict__ rows_merged, int per_warp_floats, int sort_pow2)
{
	extern __shared__ float smem[];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int64_t ray = static_cast<int64_t>(blockIdx.x) * kSamplerWarps + warp;
	if (ray >= R) return;
	const int B = S - 1;
	float* cdf = smem + static_cast<size_t>(warp) * per_warp_floats;
	float* bins = cdf + B;
	float* zs = bins + B;
	float* zc = zs + N;
	const float* zrow = z_coarse + ray * S;
	for (int k = lane; k < S; k += 32) zc[k] = zrow[k];
	__syncwarp();
	for (int k = lane; k < B; k += 32) bins[k] = 0.5f * __fadd_rn(zc[k + 1], zc[k]);  // z_vals_mid, src/NeRFRenderer.h:427
	build_cdf(weights + ray * S + 1, S - 2, cdf, lane);                                // Weights[:, 1:-1], src/NeRFRenderer.h:428
	const float* urow = u_per_ray ? u + ray * N : u;
	for (int j = lane; j < N; j += 32) {
		const float s = invert_cdf(cdf, bins, B, urow[j]);
		zs[j] = s;
		if (z_samples) z_samples[ray * N + j] = s;
	}
	__syncwarp();
	float* out = z_merged + ray * (S + N);
	if (!u_per_ray) {
		// Both lists are sorted only up to rounding: the lerp b0 + t*(b1-b0) may pass b1 by an ulp while the next sample
		// starts at b1, and for a ray that misses the box (far = near + 1e-6) near*(1-t)+far*t is not monotone in fp32.
		// Odd-even passes until clean (normally zero swaps) make the rank merge equal to torch::sort on any input.
		restore_order(zs, N, lane);
		restore_order(zc, S, lane);
		// rank merge; ties: coarse samples first
		// perm_out (optional) [R, N+S]: entry j < N is the merged position of the j-th importance sample (in sorted order); entry N+k
		// is the merged position of coarse sample k, i.e. z_merged[perm[N+k]] is bit-identical to z_coarse[r,k] — "same z, hence
		// same point": the contract the row reuse of nrf_hash_encode_rays_fwd and nrf_mlp_small_fwd_importance rely on.  With u shared
		// by the rays every entry is >= 0; the per-ray-u path below reports -(p+1) (nothing reusable).
		// rows_coarse / rows_merged (optional): the coarse pass's 16-byte raw rows [R,S,4] travel to their merged positions [R,S+N,4].
		int16_t* po = perm_out ? perm_out + ray * (S + N) : nullptr;
		bool moved = false;
		for (int k = lane; k < S; k += 32) moved |= zc[k] != zrow[k];
		if (!__any_sync(0xffffffffu, moved)) {
			for (int k = lane; k < S; k += 32) {
				const int pos = k + lower_bound(zs, N, zc[k]);
				out[pos] = zc[k];
				if (po) po[N + k] = static_cast<int16_t>(pos);
				if (rows_merged) rows_merged[ray * (S + N) + pos] = __ldg(rows_coarse + ray * S + k);
			}
		} else {
			// restore_order permuted the coarse list (a ray that misses the box): coarse sample k goes to the sorted rank of its value,
			// equal values in index order — the same merged array, and every sample keeps a position that holds its own z
			for (int k = lane; k < S; k += 32) {
				const float v = zrow[k];
				int rank = lower_bound(zc, S, v);
				for (int i = 0; i < k; i++) rank += zrow[i] == v ? 1 : 0;
				rank = min(rank, S - 1);   // only a NaN depth could get here out of range
				const int pos = rank + lower_bound(zs, N, v);
				out[pos] = v;
				if (po) po[N + k] = static_cast<int16_t>(pos);
				if (rows_merged) rows_merged[ray * (S + N) + pos] = __ldg(rows_coarse + ray * S + k);
			}
		}
		for (int j = lane; j < N; j += 32) {
			const int pos = j + upper_bound(zc, S, zs[j]);
			out[pos] = zs[j];
			if (po) po[j] = static_cast<int16_t>(pos);
		}
	} else {
		float* scratch = zc + S;
		for (int i = lane; i < sort_pow2; i += 32) scratch[i] = i < S ? zc[i] : (i < S + N ? zs[i - S] : __int_as_float(0x7f800000));
		__syncwarp();
		bitonic_sort(scratch, sort_pow2, lane);
		for (int i = lane; i < S + N; i += 32) out[i] = scratch[i];
		if (perm_out) for (int i = lane; i < S + N; i += 32) perm_out[ray * (S + N) + i] = static_cast<int16_t>(i < N ? i : -(i + 1));
	}
}

// The same, one CTA per ray (u shared by the rays).  A training batch is a few thousand rays — less than one wave of warps — so the warp-per-ray
// kernel above runs at the latency of ONE warp walking a ray's ~14 dependent binary searches per lane; here every thread owns one importance
// sample (and one coarse sample in the merge), the chain is 3 searches long; warp 0 builds the cdf (the same code, the same bits) while the
// others stage the depths.  Same arithmetic per element as
// the warp kernel: bit-identical outputs (tests/test_gpu_render.py::test_sampler_block_kernel_equals_warp_kernel).
constexpr int kSamplerBlock = 128;
constexpr int64_t kBlockPerRayMaxRays = 16384;       // about two waves of the warp-per-ray kernel

__global__ void __launch_bounds__(kSamplerBlock) sample_pdf_merge_block_kernel(const float* __restrict__ z_coarse, const float* __restrict__ weights,
	const float* __restrict__ u, int64_t R, int S, int N, float* __restrict__ z_samples, float* __restrict__ z_merged, int16_t* __restrict__ perm_out,
	const float4* __restrict__ rows_coarse, float4* __restrict__ rows_merged)
{
	extern __shared__ float smem[];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, tid = threadIdx.x;
	const int64_t ray = blockIdx.x;
	const int B = S - 1;
	float* cdf = smem;
	float* bins = cdf + B;
	float* zs = bins + B;
	float* zc = zs + N;
	const float* zrow = z_coarse + ray * S;
	if (warp == 0) build_cdf(weights + ray * S + 1, S - 2, cdf, lane);                                   // Weights[:, 1:-1], src/NeRFRenderer.h:428
	for (int k = tid; k < S; k += kSamplerBlock) zc[k] = zrow[k];
	for (int k = tid; k < B; k += kSamplerBlock) bins[k] = 0.5f * __fadd_rn(zrow[k + 1], zrow[k]);      // z_vals_mid, :427
	__syncthreads();
	for (int j = tid; j < N; j += kSamplerBlock) {
		const float s = invert_cdf(cdf, bins, B, u[j]);
		zs[j] = s;
		if (z_samples) z_samples[ray * N + j] = s;
	}
	__syncthreads();
	// restore_order on both lists (see sample_pdf_merge_kernel), CTA-wide
	for (;;) {
		int swapped = 0;
#pragma unroll
		for (int phase = 0; phase < 2; phase++) {
			for (int j = 2 * tid + phase; j + 1 < N; j += 2 * kSamplerBlock) {
				const float x = zs[j], y = zs[j + 1];
				if (x > y) { zs[j] = y; zs[j + 1] = x; swapped = 1; }
			}
			for (int j = 2 * tid + phase; j + 1 < S; j += 2 * kSamplerBlock) {
				const float x = zc[j], y = zc[j + 1];
				if (x > y) { zc[j] = y; zc[j + 1] = x; swapped = 1; }
			}
			__syncthreads();
		}
		if (!__syncthreads_or(swapped)) break;
	}
	float* out = z_merged + ray * (S + N);
	int16_t* po = perm_out ? perm_out + ray * (S + N) : nullptr;
	int moved = 0;
	for (int k = tid; k < S; k += kSamplerBlock) moved |= zc[k] != zrow[k];
	moved = __syncthreads_or(moved);
	for (int k = tid; k < S; k += kSamplerBlock) {
		float v;
		int rank;
		if (!moved) {
			v = zc[k];
			rank = k;
		} else {
			v = zrow[k];
			rank = lower_bound(zc, S, v);
			for (int i = 0; i < k; i++) rank += zrow[i] == v ? 1 : 0;
			rank = min(rank, S - 1);
		}
		const int pos = rank + lower_bound(zs, N, v);
		out[pos] = v;
		if (po) po[N + k] = static_cast<int16_t>(pos);
		if (rows_merged) rows_merged[ray * (S + N) + pos] = __ldg(rows_coarse + ray * S + k);
	}
	for (int j = tid; j < N; j += kSamplerBlock) {
		const int pos = j + upper_bound(zc, S, zs[j]);
		out[pos] = zs[j];
		if (po) po[j] = static_cast<int16_t>(pos);
	}
}

__global__ void __launch_bounds__(kSamplerWarps * 32) sample_pdf_kernel(const float* __restrict__ bins_g,
	const float* __restrict__ weights, int B, const float* __restrict__ u, int u_per_ray, int64_t R, int N,
	float* __restrict__ out)
{
	extern __shared__ float smem[];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int64_t ray = static_cast<int64_t>(blockIdx.x) * kSamplerWarps + warp;
	if (ray >= R) return;
	float* cdf = smem + static_cast<size_t>(warp) * (2 * B);
	float* bins = cdf + B;
	for (int k = lane; k < B; k += 32) bins[k] = bins_g[ray * B + k];
	build_cdf(weights + ray * (B - 1), B - 1, cdf, lane);
	const float* urow = u_per_ray ? u + ray * N : u;
	for (int j = lane; j < N; j += 32) out[ray * N + j] = invert_cdf(cdf, bins, B, urow[j]);
}

}  // namespace nrf

using namespace nrf;

extern "C" {

int nrf_sample_pdf(const float* bins, const float* weights, int32_t n_bins, const float* u, int32_t u_per_ray,
	int64_t n_rays, int32_t n_samples, float* samples_out, nrf_stream stream)
{
	NRF_REQUIRE(n_bins >= 2 && n_bins <= 1024, "n_bins out of range");
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 0, "bad sizes");
	if (n_rays == 0 || n_samples == 0) return NRF_OK;
	NRF_REQUIRE(bins && weights && u && samples_out, "null pointer");
	const unsigned blocks = static_cast<unsigned>((n_rays + kSamplerWarps - 1) / kSamplerWarps);
	const size_t smem = static_cast<size_t>(kSamplerWarps) * 2 * n_bins * sizeof(float);
	sample_pdf_kernel<<<blocks, kSamplerWarps * 32, smem, as_stream(stream)>>>(bins, weights, n_bins, u, u_per_ray, n_rays, n_samples, samples_out);
	NRF_CHECK_LAUNCH("sample_pdf_kernel");
	return NRF_OK;
}

int nrf_sample_pdf_merge(const float* z_coarse, const float* weights, const float* u, int32_t u_per_ray, int64_t n_rays,
	int32_t n_samples, int32_t n_importance, float* z_samples, float* z_merged, nrf_stream stream)
{
	return nrf_sample_pdf_merge_perm(z_coarse, weights, u, u_per_ray, n_rays, n_samples, n_importance, z_samples, z_merged, nullptr, stream);
}

int nrf_sample_pdf_merge_perm(const float* z_coarse, const float* weights, const float* u, int32_t u_per_ray, int64_t n_rays,
	int32_t n_samples, int32_t n_importance, float* z_samples, float* z_merged, int16_t* perm_out, nrf_stream stream)
{
	return nrf_sample_pdf_merge_rows(z_coarse, weights, u, u_per_ray, n_rays, n_samples, n_importance, z_samples, z_merged, perm_out, nullptr, nullptr,
		stream);
}

int nrf_sample_pdf_merge_rows(const float* z_coarse, const float* weights, const float* u, int32_t u_per_ray, int64_t n_rays,
	int32_t n_samples, int32_t n_importance, float* z_samples, float* z_merged, int16_t* perm_out, const float* rows_coarse, float* rows_merged,
	nrf_stream stream)
{
	NRF_REQUIRE(n_samples >= 3, "n_samples must be >= 3");
	NRF_REQUIRE(n_importance >= 1, "n_importance must be >= 1");
	NRF_REQUIRE(n_samples + n_importance <= 1024, "n_samples + n_importance > 1024");
	NRF_REQUIRE(n_rays >= 0, "bad sizes");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(z_coarse && weights && u && z_merged, "null pointer");
	NRF_REQUIRE((rows_coarse == nullptr) == (rows_merged == nullptr), "rows_coarse and rows_merged go together");
	NRF_REQUIRE(!rows_merged || !u_per_ray, "the raw-row scatter needs u shared by the rays (per-ray u re-sorts: nothing is reusable)");
	NRF_REQUIRE(((reinterpret_cast<uintptr_t>(rows_coarse) | reinterpret_cast<uintptr_t>(rows_merged)) & 15) == 0, "raw rows must be 16-byte aligned");
	int pow2 = 1;
	while (pow2 < n_samples + n_importance) pow2 <<= 1;
	const int per_warp = 2 * (n_samples - 1) + n_importance + n_samples + (u_per_ray ? pow2 : 0);
	const size_t smem = static_cast<size_t>(kSamplerWarps) * per_warp * sizeof(float);
	NRF_REQUIRE(smem <= 48 * 1024, "shared memory budget exceeded");
	// few rays (a training batch): one CTA per ray, latency of 3 searches instead of 14; many rays (a render chunk) or per-ray u: one warp
	// per ray, fewer instructions per ray
	const bool per_block = !u_per_ray && n_rays <= kBlockPerRayMaxRays;
	if (per_block) {
		const size_t smem_b = static_cast<size_t>(2 * (n_samples - 1) + n_importance + n_samples) * sizeof(float);
		sample_pdf_merge_block_kernel<<<static_cast<unsigned>(n_rays), kSamplerBlock, smem_b, as_stream(stream)>>>(z_coarse, weights, u, n_rays,
			n_samples, n_importance, z_samples, z_merged, perm_out, reinterpret_cast<const float4*>(rows_coarse), reinterpret_cast<float4*>(rows_merged));
		NRF_CHECK_LAUNCH("sample_pdf_merge_block_kernel");
		return NRF_OK;
	}
	const unsigned blocks = static_cast<unsigned>((n_rays + kSamplerWarps - 1) / kSamplerWarps);
	sample_pdf_merge_kernel<<<blocks, kSamplerWarps * 32, smem, as_stream(stream)>>>(z_coarse, weights, u, u_per_ray, n_rays,
		n_samples, n_importance, z_samples, z_merged, perm_out, reinterpret_cast<const float4*>(rows_coarse), reinterpret_cast<float4*>(rows_merged),
		per_warp, pow2);
	NRF_CHECK_LAUNCH("sample_pdf_merge_kernel");
	return NRF_OK;
}

}
