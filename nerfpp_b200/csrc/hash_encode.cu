// Multiresolution hash-grid encode, forward and backward, for sm_100a.
//
// Replaces CuHashEmbedderForwardKernel / CuHashEmbedderBackwardKernel and their host wrappers
// (reference src/CuHashEmbedder.cu:9-102, 106-216, 221-325) plus the clamp / keep-mask prologue of
// CuHashEmbedderImpl::forward (src/CuHashEmbedder.cpp:85-103).
//
// Index arithmetic is bit-exact with the reference: same device expression for the per-level scale
// (precomputed once by nrf_hash_level_scales), IEEE division for the box normalisation, uint32 wrap-around
// multiply/xor, `% size`, and the reference's scalar (not row) level offsets (SURVEY §9-Q6/Q7).
//
// B200 layout choices (vs the reference's one thread per (point, level), grid.y = level):
//   * one thread per POINT walks all levels: the point is read and normalised once, the 8 gathers of a level
//     are issued back to back (8..32 loads in flight per thread), and the L*F outputs of a point leave as
//     16-byte vector stores instead of 4-byte stores at 64-byte stride;
//   * the table is the persistent fp16 shadow (17 MiB used at the BASELINE shape, L2 resident) kept up to date
//     by nrf_adam_step, not a per-call cast of the fp32 master;
//   * level metadata (scale, primes, offsets) is staged once per CTA in shared memory;
//   * the backward accumulates in fp32 with vector RED (red.global.add.v2.f32), no x128 loss scale.
#include "common.cuh"
#include "jitter.cuh"
#include <string.h>

namespace nrf {

struct HashMeta {
	float scale[NRF_MAX_LEVELS];
	float bx[NRF_MAX_LEVELS], by[NRF_MAX_LEVELS], bz[NRF_MAX_LEVELS];
	uint32_t pa[NRF_MAX_LEVELS], pb[NRF_MAX_LEVELS], pc[NRF_MAX_LEVELS];
	uint32_t offset[NRF_MAX_LEVELS], size[NRF_MAX_LEVELS], mask[NRF_MAX_LEVELS];
	// x % size without a division (Granlund & Montgomery, unsigned division by an invariant): t = umulhi(x, magic),
	// q = (t + ((x - t) >> 1)) >> shift, x - q * size.  shift == kPow2 marks a power-of-two size: x & mask instead.
	uint32_t magic[NRF_MAX_LEVELS], shift[NRF_MAX_LEVELS];
};
constexpr uint32_t kPow2 = 32u;

struct HashArgs {
	int n_levels, n_volumes;
	float min_x, min_y, min_z, max_x, max_y, max_z;
	const int32_t* primes;
	const float* biases;
	const int32_t* feat_local_idx;
	const int32_t* feat_local_size;
	const float* level_scale;
};

__device__ __forceinline__ void stage_meta(HashMeta& m, const HashArgs& a)
{
	for (int l = threadIdx.x; l < a.n_levels; l += blockDim.x) {
		const int t = l * a.n_volumes;  // volume index is always 0 (src/CuHashEmbedder.cpp:97)
		m.scale[l] = a.level_scale[l];
		m.pa[l] = static_cast<uint32_t>(a.primes[t * 3 + 0]);
		m.pb[l] = static_cast<uint32_t>(a.primes[t * 3 + 1]);
		m.pc[l] = static_cast<uint32_t>(a.primes[t * 3 + 2]);
		m.bx[l] = a.biases[t * 3 + 0];
		m.by[l] = a.biases[t * 3 + 1];
		m.bz[l] = a.biases[t * 3 + 2];
		m.offset[l] = static_cast<uint32_t>(a.feat_local_idx[l]);
		const uint32_t sz = static_cast<uint32_t>(a.feat_local_size[l]);
		m.size[l] = sz;
		if ((sz & (sz - 1u)) == 0u) {
			m.mask[l] = sz - 1u; m.magic[l] = 0u; m.shift[l] = kPow2;
		} else {
			const uint32_t lg = 32u - static_cast<uint32_t>(__clz(sz - 1u));                    // ceil(log2 size), size >= 3 here
			m.mask[l] = 0u;
			m.magic[l] = static_cast<uint32_t>((((1ull << lg) - sz) << 32) / sz + 1ull);
			m.shift[l] = lg - 1u;
		}
	}
	__syncthreads();
}

// Same expression as src/CuHashEmbedder.cu:40, evaluated on the device so that the rounding is the device's.
__global__ void level_scale_kernel(int base_resolution, int finest_resolution, int n_levels, float* out)
{
	const int level_idx = threadIdx.x;
	if (level_idx >= n_levels) return;
	out[level_idx] = exp2f((log2f(finest_resolution) - log2f(base_resolution)) * float(level_idx) / float(n_levels - 1) + log2f(base_resolution));
}

// Where the sample points come from: an explicit [N,3] array, or — fused point generation, src/NeRFRenderer.h:419,432 —
// pts = o + d * z evaluated here from the ray batch and the z values with ATen's un-fused rounding (mul, then add), so the
// cells are those of the reference's materialised points and the [R,S,3] array never exists.
struct PointSrc {
	const float* points;      // [N,3] or nullptr
	const float* ray_batch;   // [R, ray_stride]: o at 0..2, d at 3..5
	const float* z;           // [R,S]
	int ray_stride, S;
	// forward only: work items run (ray tile, sample, ray in tile) instead of (ray, sample) when group > 1, so that neighbouring lanes hold
	// the SAME sample of `group` neighbouring rays — for the rays of a rendered frame (adjacent pixels) these points lie a fraction of a
	// fine cell apart and share most of their corner fetches, while consecutive samples of one ray are cells apart.  Results do not change.
	int group, R;
	int S_work;       // samples per ray the grouped order enumerates: S, or (row reuse without a copy) the importance samples only
};

__device__ __forceinline__ void load_point(const PointSrc& ps, int64_t i, float& x, float& y, float& z)
{
	if (ps.points) {
		x = ps.points[i * 3 + 0]; y = ps.points[i * 3 + 1]; z = ps.points[i * 3 + 2];
	} else {
		const uint32_t ray = static_cast<uint32_t>(i) / static_cast<uint32_t>(ps.S);   // N < 2^31 checked by the host
		const float* rb = ps.ray_batch + static_cast<int64_t>(ray) * ps.ray_stride;
		const float zi = ps.z[i];
		x = __fadd_rn(__ldg(rb + 0), __fmul_rn(__ldg(rb + 3), zi));
		y = __fadd_rn(__ldg(rb + 1), __fmul_rn(__ldg(rb + 4), zi));
		z = __fadd_rn(__ldg(rb + 2), __fmul_rn(__ldg(rb + 5), zi));
	}
}

// The same rays with the per-sample perturbations of the reference's shipped training configuration (nrf_point_jitter), applied in the
// order of src/NeRFRenderer.h:419-445: p = o + d z; [sp_noise] ReflectBoundary(p + noise * alpha) (:435-443); [cone] += TangentScatter
// offset (:307-362), clamped into the box if asked (:356-360).  jitter.cuh holds the arithmetic, shared with nrf_tangent_scatter /
// nrf_precondition_points, so the points are those the composed path materialises, bit for bit.  No row reuse, no ray grouping.
struct JitterSrc {
	const float* ray_batch;
	const float* z;
	int ray_stride, S;
	const float* cone;
	int cone_stride;
	const float* rand_r;
	const float* rand_theta;
	int clamp_box;
	const float* sp_noise;
	const float* sp_alpha;
	Box box;
	static constexpr int group = 1, R = 0, S_work = 0;
};

__device__ __forceinline__ void load_point(const JitterSrc& ps, int64_t i, float& x, float& y, float& z)
{
	const uint32_t ray = static_cast<uint32_t>(i) / static_cast<uint32_t>(ps.S);   // N < 2^31 checked by the host
	const float* rb = ps.ray_batch + static_cast<int64_t>(ray) * ps.ray_stride;
	const float zi = ps.z[i];
	const float dx = __ldg(rb + 3), dy = __ldg(rb + 4), dz = __ldg(rb + 5);
	x = __fadd_rn(__ldg(rb + 0), __fmul_rn(dx, zi));
	y = __fadd_rn(__ldg(rb + 1), __fmul_rn(dy, zi));
	z = __fadd_rn(__ldg(rb + 2), __fmul_rn(dz, zi));
	if (ps.sp_noise) {
		const float alpha = __ldg(ps.sp_alpha);
		const float* nz = ps.sp_noise + i * 3;
		x = precondition_coord(x, __ldg(nz + 0), alpha, ps.box.lo[0], ps.box.hi[0]);
		y = precondition_coord(y, __ldg(nz + 1), alpha, ps.box.lo[1], ps.box.hi[1]);
		z = precondition_coord(z, __ldg(nz + 2), alpha, ps.box.lo[2], ps.box.hi[2]);
	}
	if (ps.cone) {
		float off[3];
		tangent_direction(dx, dy, dz, __ldg(ps.rand_r + i), __ldg(ps.rand_theta + i), off);
		const float radius = __fmul_rn(__ldg(ps.cone + (ps.cone_stride ? static_cast<int64_t>(ray) * ps.cone_stride : 0)), zi);
		apply_tangent_offset(off, radius, x, y, z);
		if (ps.clamp_box) clamp_to_box(ps.box, x, y, z);
	}
}

// Rows of the fine pass that are bit-identical to rows the coarse pass already encoded (same z => same point => same
// cells, same table).  perm [R, N+S_prev] is nrf_sample_pdf_merge_perm's output: thread t of a ray handles
//   t <  N          the t-th importance sample: encode it, write row perm[t]
//   t >= N, p >= 0  coarse sample t-N, found unchanged at merged position p: COPY its row (and keep flag) from the coarse pass
//                   (enc == nullptr: leave the row alone — inference, where nrf_mlp_small_fwd_importance never reads it)
//   t >= N, p <  0  coarse sample whose z moved: encode the merged position -(p+1) like any other
// so that warps are homogeneous (all-encode or all-copy) instead of one lane in three idling through every gather.
struct Reuse {
	const int16_t* perm;      // [R, S] (S = N + S_prev) or nullptr
	const void* enc;          // [R, S_prev, L*F] in the output layout, or nullptr = do not copy
	const uint8_t* keep;      // [R, S_prev] or nullptr
	int S_prev;
};

struct Cell {
	uint32_t pos[8];
	float w[8];
	uint32_t cx, cy, cz;   // integer cell of the point at this level (identifies the 8 corners; the backward's run key)
};

// src/CuHashEmbedder.cu:44-90 for one level.  q = (pt - box_min) / (box_max - box_min) is level independent.
__device__ __forceinline__ void locate(const HashMeta& m, int l, float qx, float qy, float qz, Cell& c)
{
	float px = qx * m.scale[l];
	float py = qy * m.scale[l];
	float pz = qz * m.scale[l];
	px += m.bx[l];
	py += m.by[l];
	pz += m.bz[l];
	const float fx = floorf(px), fy = floorf(py), fz = floorf(pz);
	const uint32_t pos_x = static_cast<uint32_t>(fx);
	const uint32_t pos_y = static_cast<uint32_t>(fy);
	const uint32_t pos_z = static_cast<uint32_t>(fz);
	c.cx = pos_x; c.cy = pos_y; c.cz = pos_z;
	const uint32_t pa = m.pa[l], pb = m.pb[l], pc = m.pc[l];
	const uint32_t x0 = pos_x * pa, x1 = (pos_x + 1u) * pa;
	const uint32_t y0 = pos_y * pb, y1 = (pos_y + 1u) * pb;
	const uint32_t z0 = pos_z * pc, z1 = (pos_z + 1u) * pc;
	c.pos[0] = x0 ^ y0 ^ z0;
	c.pos[1] = x0 ^ y0 ^ z1;
	c.pos[2] = x0 ^ y1 ^ z0;
	c.pos[3] = x0 ^ y1 ^ z1;
	c.pos[4] = x1 ^ y0 ^ z0;
	c.pos[5] = x1 ^ y0 ^ z1;
	c.pos[6] = x1 ^ y1 ^ z0;
	c.pos[7] = x1 ^ y1 ^ z1;
	const uint32_t sh = m.shift[l];
	if (sh == kPow2) {
		const uint32_t mask = m.mask[l];
#pragma unroll
		for (int d = 0; d < 8; d++) c.pos[d] &= mask;
	} else {
		const uint32_t sz = m.size[l], mg = m.magic[l];
#pragma unroll
		for (int d = 0; d < 8; d++) {
			const uint32_t x = c.pos[d], t = __umulhi(x, mg);
			c.pos[d] = x - ((t + ((x - t) >> 1)) >> sh) * sz;                                     // == x % sz, every x
		}
	}
	const float a = px - fx, b = py - fy, cc = pz - fz;
	c.w[0] = (1.f - a) * (1.f - b) * (1.f - cc);
	c.w[1] = (1.f - a) * (1.f - b) * cc;
	c.w[2] = (1.f - a) * b * (1.f - cc);
	c.w[3] = (1.f - a) * b * cc;
	c.w[4] = a * (1.f - b) * (1.f - cc);
	c.w[5] = a * (1.f - b) * cc;
	c.w[6] = a * b * (1.f - cc);
	c.w[7] = a * b * cc;
}

// Clamp into the box and report whether the point was inside (src/CuHashEmbedder.cpp:92-94,101).
__device__ __forceinline__ bool clamp_point(const HashArgs& a, float& x, float& y, float& z)
{
	const float cx = fmaxf(fminf(x, a.max_x), a.min_x);
	const float cy = fmaxf(fminf(y, a.max_y), a.min_y);
	const float cz = fmaxf(fminf(z, a.max_z), a.min_z);
	const bool keep = (x == cx) && (y == cy) && (z == cz);
	x = cx; y = cy; z = cz;
	return keep;
}

template <int F> struct FeatVec;
template <> struct FeatVec<2> { using type = uint32_t; };
template <> struct FeatVec<4> { using type = uint2; };
template <> struct FeatVec<8> { using type = uint4; };

template <int F>
__device__ __forceinline__ void unpack(const typename FeatVec<F>::type& v, float (&f)[F])
{
	const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
	for (int k = 0; k < F / 2; k++) {
		const float2 t = __half22float2(h[k]);
		f[2 * k] = t.x;
		f[2 * k + 1] = t.y;
	}
}

// F features per level; CH = levels handled per 16-byte output chunk (8 halves).
//
// Work item = (point, part).  SPLIT == 1: one thread walks all levels of its point.  SPLIT == number of chunks (4 at L16 F2): SPLIT
// neighbouring lanes share a point and each handles ONE chunk of CH levels, so a warp writes 32 / SPLIT complete rows as one contiguous
// block and an item is 1 / SPLIT of the dependent-latency chain.  Every thread handles `iters` items at a stride of the whole grid: the
// launch passes iters = 1 (one item per thread; see launch_plan for the persistent-grid experiment that was not kept).
template <int F, bool OUT_F32, int SPLIT, class PS>
__device__ __forceinline__ void hash_fwd_body(const HashArgs& a, const __half* __restrict__ table,
	const PS& ps, const Reuse& ru, int64_t n_items, int64_t stride, int iters, int clamp_points, uint8_t* __restrict__ keep, void* __restrict__ out)
{
	constexpr int CH = 8 / F;
	using V = typename FeatVec<F>::type;
	__shared__ HashMeta m;
	stage_meta(m, a);
	const int L = a.n_levels;
	const int row_bytes = L * F * (OUT_F32 ? 4 : 2);

	int64_t item = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	for (int it = 0; it < iters; it++, item += stride) {
		if (item >= n_items) break;
		int64_t i = SPLIT == 1 ? item : item / SPLIT;
		const int part = SPLIT == 1 ? 0 : static_cast<int>(item & (SPLIT - 1));
		if (ps.group > 1) {
			// (ray tile, sample, ray in tile); only the first S_work samples of a ray are enumerated.  MEASURED AND NOT KEPT
			// (profiles/r2_render_ray_group_sweep.jsonl): lanes = 32 neighbouring rays with the level chunk warp-uniform, so that one gather
			// instruction covers 32 rays at ONE level — 54.9 ms / C4 frame against 50.6 ms with SPLIT lanes per point.
			const uint32_t per = static_cast<uint32_t>(ps.group) * static_cast<uint32_t>(ps.S_work);
			const uint32_t tile = static_cast<uint32_t>(i) / per, rem = static_cast<uint32_t>(i) - tile * per;
			const uint32_t smp = rem / static_cast<uint32_t>(ps.group), ray = tile * ps.group + (rem - smp * ps.group);
			if (ray >= static_cast<uint32_t>(ps.R)) continue;
			i = static_cast<int64_t>(ray) * ps.S + smp;
		}

		if (ru.perm) {
			const uint32_t ray = static_cast<uint32_t>(i) / static_cast<uint32_t>(ps.S);
			const int t = static_cast<int>(static_cast<uint32_t>(i) - ray * static_cast<uint32_t>(ps.S));
			const int p = ru.perm[i];
			const int64_t row0 = static_cast<int64_t>(ray) * ps.S;
			if (p >= 0 && t >= ps.S - ru.S_prev) {
				// copy the row the coarse pass produced for this very point (16-byte vectors; rows are 16-byte aligned, host-checked)
				const int64_t from = static_cast<int64_t>(ray) * ru.S_prev + (t - (ps.S - ru.S_prev));
				const uint4* s4 = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(ru.enc) + from * row_bytes);
				uint4* d4 = reinterpret_cast<uint4*>(reinterpret_cast<char*>(out) + (row0 + p) * row_bytes);
				const int nq = ru.enc ? row_bytes / 16 : 0;   // enc == nullptr: the caller reads these rows nowhere (inference), skip the copy
				if (SPLIT == 1) {
					for (int q = 0; q < nq; q++) d4[q] = __ldg(s4 + q);
				} else {
					for (int q = part; q < nq; q += SPLIT) d4[q] = __ldg(s4 + q);
				}
				if (keep && part == 0) keep[row0 + p] = ru.keep ? ru.keep[from] : 1;
				continue;
			}
			i = row0 + (p >= 0 ? p : -(p + 1));   // the merged position this thread encodes
		}

		float x, y, z;
		load_point(ps, i, x, y, z);
		if (clamp_points) {
			const bool k = clamp_point(a, x, y, z);
			if (keep && part == 0) keep[i] = k ? 1 : 0;
		}
		const float qx = (x - a.min_x) / (a.max_x - a.min_x);
		const float qy = (y - a.min_y) / (a.max_y - a.min_y);
		const float qz = (z - a.min_z) / (a.max_z - a.min_z);

		const int64_t row = i * (static_cast<int64_t>(L) * F);
		const int l_begin = SPLIT == 1 ? 0 : part * CH;
		const int l_end = SPLIT == 1 ? L : min(L, l_begin + CH);
		for (int l0 = l_begin; l0 < l_end; l0 += CH) {
			__half2 acc[4];
#pragma unroll
			for (int j = 0; j < CH; j++) {
				const int l = l0 + j;
				if (l < L) {
					Cell c;
					locate(m, l, qx, qy, qz, c);
					const __half* base = table + m.offset[l];
					V v[8];
#pragma unroll
					for (int d = 0; d < 8; d++) v[d] = __ldg(reinterpret_cast<const V*>(base + static_cast<size_t>(c.pos[d]) * F));
					float f[8][F];
#pragma unroll
					for (int d = 0; d < 8; d++) unpack<F>(v[d], f[d]);
#pragma unroll
					for (int k = 0; k < F; k += 2) {
						// same summation order as src/CuHashEmbedder.cu:96-100
						const float r0 = c.w[0] * f[0][k] + c.w[1] * f[1][k] + c.w[2] * f[2][k] + c.w[3] * f[3][k] +
						                 c.w[4] * f[4][k] + c.w[5] * f[5][k] + c.w[6] * f[6][k] + c.w[7] * f[7][k];
						const float r1 = c.w[0] * f[0][k + 1] + c.w[1] * f[1][k + 1] + c.w[2] * f[2][k + 1] + c.w[3] * f[3][k + 1] +
						                 c.w[4] * f[4][k + 1] + c.w[5] * f[5][k + 1] + c.w[6] * f[6][k + 1] + c.w[7] * f[7][k + 1];
						acc[(j * F + k) / 2] = __halves2half2(__float2half_rn(r0), __float2half_rn(r1));
					}
				} else {
#pragma unroll
					for (int k = 0; k < F; k += 2) acc[(j * F + k) / 2] = __halves2half2(__half(0), __half(0));
				}
			}
			const int n_valid = min(CH, L - l0) * F;  // scalars of this chunk that exist
			if (OUT_F32) {
				float* o = reinterpret_cast<float*>(out) + row + static_cast<int64_t>(l0) * F;
				float v8[8];
#pragma unroll
				for (int k = 0; k < 4; k++) {
					const float2 t = __half22float2(acc[k]);
					v8[2 * k] = t.x;
					v8[2 * k + 1] = t.y;
				}
				if (n_valid == 8 && ((L * F) % 4 == 0)) {
					reinterpret_cast<float4*>(o)[0] = make_float4(v8[0], v8[1], v8[2], v8[3]);
					reinterpret_cast<float4*>(o)[1] = make_float4(v8[4], v8[5], v8[6], v8[7]);
				} else {
					for (int k = 0; k < n_valid; k++) o[k] = v8[k];
				}
			} else {
				__half* o = reinterpret_cast<__half*>(out) + row + static_cast<int64_t>(l0) * F;
				if (n_valid == 8 && ((L * F) % 8 == 0)) {
					*reinterpret_cast<uint4*>(o) = *reinterpret_cast<const uint4*>(acc);
				} else {
					const __half* hs = reinterpret_cast<const __half*>(acc);
					for (int k = 0; k < n_valid; k++) o[k] = hs[k];
				}
			}
		}
	}
}

template <int F, bool OUT_F32, int SPLIT>
__global__ void __launch_bounds__(128) hash_fwd_kernel(HashArgs a, const __half* __restrict__ table,
	PointSrc ps, Reuse ru, int64_t n_items, int64_t stride, int iters, int clamp_points, uint8_t* __restrict__ keep, void* __restrict__ out)
{
	hash_fwd_body<F, OUT_F32, SPLIT>(a, table, ps, ru, n_items, stride, iters, clamp_points, keep, out);
}

// a separate instantiation, so that the parity kernels above keep their code; `ru` (same launch signature) is not read: no row reuse
template <int F, bool OUT_F32, int SPLIT>
__global__ void __launch_bounds__(128) hash_fwd_jitter_kernel(HashArgs a, const __half* __restrict__ table,
	JitterSrc ps, Reuse ru, int64_t n_items, int64_t stride, int iters, int clamp_points, uint8_t* __restrict__ keep, void* __restrict__ out)
{
	hash_fwd_body<F, OUT_F32, SPLIT>(a, table, ps, Reuse{nullptr, nullptr, nullptr, 0}, n_items, stride, iters, clamp_points, keep, out);
}

__device__ __forceinline__ void red_add_v2(float* addr, float a, float b)
{
	asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b) : "memory");
}

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d)
{
	asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Backward: dTable[corner] += w_corner * dEnc, fp32 RED (src/CuHashEmbedder.cu:106-216).
//
// Warp-aggregated scatter.  Points arrive in ray-major order (samples of a ray are consecutive), so on the coarse levels
// neighbouring lanes of a warp sit in the SAME grid cell and would hit the same 8 table entries.  Per level the warp
//   1. flags lanes whose cell equals the previous lane's cell (3 SHFL + 1 ballot) -> contiguous runs of equal cells,
//   2. sums the 8 x F corner contributions over each run with a segmented shuffle reduction whose depth is chosen from the
//      longest run in the warp (warp-uniform; zero steps on the fine levels where every lane is alone in its cell),
//   3. lets only the first lane of a run issue the vector REDs.
// Any point order is handled correctly (a run is defined by adjacency, not by key equality); ray-major order is what
// makes it pay.  The reference issues N*L*8 half2 atomics regardless (SURVEY §8a-a3).
// Thread t handles points t, t + stride, ... (`iters` of them, warp-uniform; the launch passes iters = 1).
template <int F, bool GRAD_BF16, class PS>
__device__ __forceinline__ void hash_bwd_body(HashArgs a, PS ps, int64_t n_points, int64_t stride, int iters,
	int clamp_points, const void* __restrict__ grad_enc, float* __restrict__ grad_table)
{
	constexpr int CH = 8 / F;   // levels per 8-value gradient chunk (16 B of bf16 / 32 B of fp32)
	constexpr uint32_t FULL = 0xffffffffu;
	__shared__ HashMeta m;
	stage_meta(m, a);

	const int lane = threadIdx.x & 31;
	int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	for (int it = 0; it < iters; it++, i += stride) {
	const bool valid = i < n_points;   // no early return: the whole warp takes part in the shuffles

	float x = 0.f, y = 0.f, z = 0.f;
	if (valid) load_point(ps, i, x, y, z);
	if (clamp_points) clamp_point(a, x, y, z);
	const float qx = (x - a.min_x) / (a.max_x - a.min_x);
	const float qy = (y - a.min_y) / (a.max_y - a.min_y);
	const float qz = (z - a.min_z) / (a.max_z - a.min_z);

	const int L = a.n_levels;
	const int D = L * F;
	const int64_t row = i * static_cast<int64_t>(D);
	const bool vec_ok = (D % 8) == 0;   // rows are 16-byte (bf16) / 32-byte (fp32) aligned
	for (int l0 = 0; l0 < L; l0 += CH) {
		float g8[8];
#pragma unroll
		for (int k = 0; k < 8; k++) g8[k] = 0.f;
		if (valid) {
			const int n_valid = min(CH, L - l0) * F;
			if (GRAD_BF16) {
				const __nv_bfloat16* gp = reinterpret_cast<const __nv_bfloat16*>(grad_enc) + row + static_cast<int64_t>(l0) * F;
				if (vec_ok) {
					const uint4 v = __ldg(reinterpret_cast<const uint4*>(gp));
					const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
					for (int k = 0; k < 4; k++) {
						const float2 t = __bfloat1622float2(h[k]);
						g8[2 * k] = t.x;
						g8[2 * k + 1] = t.y;
					}
				} else {
#pragma unroll
					for (int k = 0; k < 8; k++) if (k < n_valid) g8[k] = __bfloat162float(gp[k]);
				}
			} else {
				const float* gp = reinterpret_cast<const float*>(grad_enc) + row + static_cast<int64_t>(l0) * F;
				if (vec_ok) {
					const float4 v0 = __ldg(reinterpret_cast<const float4*>(gp)), v1 = __ldg(reinterpret_cast<const float4*>(gp) + 1);
					g8[0] = v0.x; g8[1] = v0.y; g8[2] = v0.z; g8[3] = v0.w;
					g8[4] = v1.x; g8[5] = v1.y; g8[6] = v1.z; g8[7] = v1.w;
				} else {
#pragma unroll
					for (int k = 0; k < 8; k++) if (k < n_valid) g8[k] = gp[k];
				}
			}
		}
		const int jn = min(CH, L - l0);   // levels of this chunk (warp-uniform)
		for (int j = 0; j < jn; j++) {
			const int l = l0 + j;
			float g[F];
			bool any = false;
#pragma unroll
			for (int k = 0; k < F; k++) {
				g[k] = g8[k];
				any |= (g[k] != 0.f);
			}
#pragma unroll
			for (int k = 0; k + F < 8; k++) g8[k] = g8[k + F];   // next level's values move to the front (static indices only)
			const bool active = valid && any;   // src/CuHashEmbedder.cu:195 skips all-zero gradients
			Cell c;
			locate(m, l, qx, qy, qz, c);
			// ---- runs of equal cells among neighbouring active lanes
			const uint32_t px_ = __shfl_up_sync(FULL, c.cx, 1), py_ = __shfl_up_sync(FULL, c.cy, 1), pz_ = __shfl_up_sync(FULL, c.cz, 1);
			const bool prev_active = __shfl_up_sync(FULL, static_cast<int>(active), 1) != 0;
			const bool cont = lane > 0 && active && prev_active && px_ == c.cx && py_ == c.cy && pz_ == c.cz;
			const uint32_t nh = __ballot_sync(FULL, cont);   // bit j: lane j continues lane j-1's run
			if (__ballot_sync(FULL, active) == 0u) continue;  // warp-uniform
			float v[8][F];
#pragma unroll
			for (int d = 0; d < 8; d++)
#pragma unroll
				for (int k = 0; k < F; k++) v[d][k] = g[k] * c.w[d];
			if (nh != 0u) {
				// depth of the segmented reduction from the longest run: > 2^s lanes <=> 2^s consecutive continuation bits
				const uint32_t t2 = nh & (nh >> 1), t4 = t2 & (t2 >> 2), t8 = t4 & (t4 >> 4), t16 = t8 & (t8 >> 8);
				const int steps = 1 + (t2 != 0u) + (t4 != 0u) + (t8 != 0u) + (t16 != 0u);
				const uint32_t above = lane < 31 ? (nh >> (lane + 1)) : 0u;   // bit b: lane+1+b continues its predecessor
				for (int s = 0; s < steps; s++) {   // warp-uniform trip count
					const int off = 1 << s;
					// lane+off is in my run  <=>  lanes lane+1 .. lane+off all continue their predecessor
					const uint32_t need = (off == 32) ? FULL : ((1u << off) - 1u);
					const bool take = (lane + off < 32) && ((above & need) == need);
#pragma unroll
					for (int d = 0; d < 8; d++)
#pragma unroll
						for (int k = 0; k < F; k++) {
							const float o = __shfl_down_sync(FULL, v[d][k], off);
							if (take) v[d][k] += o;
						}
				}
			}
			if (active && !cont) {   // first lane of a run owns the run's sum
				float* base = grad_table + m.offset[l];
				const bool vec4_ok = (reinterpret_cast<uintptr_t>(base) & 15) == 0;
#pragma unroll
				for (int d = 0; d < 8; d++) {
					float* p = base + static_cast<size_t>(c.pos[d]) * F;
					if (F % 4 == 0 && vec4_ok) {
						// an entry of F >= 4 features is 16-byte aligned when the level offset is: half as many L2 atomic operations
#pragma unroll
						for (int k = 0; k + 3 < F; k += 4) red_add_v4(p + k, v[d][k], v[d][k + 1], v[d][k + 2], v[d][k + 3]);
					} else {
#pragma unroll
						for (int k = 0; k < F; k += 2) red_add_v2(p + k, v[d][k], v[d][k + 1]);
					}
				}
			}
		}
	}
	}   // items of this thread
}

template <int F, bool GRAD_BF16>
__global__ void __launch_bounds__(128) hash_bwd_kernel(HashArgs a, PointSrc ps, int64_t n_points, int64_t stride, int iters,
	int clamp_points, const void* __restrict__ grad_enc, float* __restrict__ grad_table)
{
	hash_bwd_body<F, GRAD_BF16>(a, ps, n_points, stride, iters, clamp_points, grad_enc, grad_table);
}

template <int F, bool GRAD_BF16>
__global__ void __launch_bounds__(128) hash_bwd_jitter_kernel(HashArgs a, JitterSrc ps, int64_t n_points, int64_t stride, int iters,
	int clamp_points, const void* __restrict__ grad_enc, float* __restrict__ grad_table)
{
	hash_bwd_body<F, GRAD_BF16>(a, ps, n_points, stride, iters, clamp_points, grad_enc, grad_table);
}

// kernel of a point source, for the launch code shared by both
template <int F, bool O, int SP> auto fwd_kernel(const PointSrc&) { return hash_fwd_kernel<F, O, SP>; }
template <int F, bool O, int SP> auto fwd_kernel(const JitterSrc&) { return hash_fwd_jitter_kernel<F, O, SP>; }
template <int F, bool G> auto bwd_kernel(const PointSrc&) { return hash_bwd_kernel<F, G>; }
template <int F, bool G> auto bwd_kernel(const JitterSrc&) { return hash_bwd_jitter_kernel<F, G>; }

// Inspection entry (tests): the scalar addresses and trilinear weights the encode kernels use, from the SAME clamp_point / locate code.
__global__ void __launch_bounds__(128) hash_cells_kernel(HashArgs a, const float* __restrict__ points, int64_t n_points, int clamp_points,
	int n_features, int64_t* __restrict__ addr, float* __restrict__ weights)
{
	__shared__ HashMeta m;
	stage_meta(m, a);
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n_points) return;
	float x = points[i * 3 + 0], y = points[i * 3 + 1], z = points[i * 3 + 2];
	if (clamp_points) clamp_point(a, x, y, z);
	const float qx = (x - a.min_x) / (a.max_x - a.min_x);
	const float qy = (y - a.min_y) / (a.max_y - a.min_y);
	const float qz = (z - a.min_z) / (a.max_z - a.min_z);
	for (int l = 0; l < a.n_levels; l++) {
		Cell c;
		locate(m, l, qx, qy, qz, c);
		for (int d = 0; d < 8; d++) {
			const int64_t o = (i * a.n_levels + l) * 8 + d;
			addr[o] = static_cast<int64_t>(m.offset[l]) + static_cast<int64_t>(c.pos[d]) * n_features;
			weights[o] = c.w[d];
		}
	}
}

__global__ void __launch_bounds__(256) table_to_half_kernel(const float* __restrict__ src, __half* __restrict__ dst, int64_t n)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x * 4;
	for (int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
		if (i + 3 < n) {
			const float4 v = *reinterpret_cast<const float4*>(src + i);
			__half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
			uint2 o;
			o.x = *reinterpret_cast<uint32_t*>(&lo);
			o.y = *reinterpret_cast<uint32_t*>(&hi);
			*reinterpret_cast<uint2*>(dst + i) = o;
		} else {
			for (int64_t j = i; j < n; j++) dst[j] = __float2half_rn(src[j]);
		}
	}
}

static int fill_args(const nrf_hash_grid* g, HashArgs& a)
{
	NRF_REQUIRE(g != nullptr, "grid is null");
	NRF_REQUIRE(g->n_levels >= 1 && g->n_levels <= NRF_MAX_LEVELS, "n_levels out of range");
	NRF_REQUIRE(g->n_volumes >= 1, "n_volumes must be >= 1");
	NRF_REQUIRE(g->primes && g->biases && g->feat_local_idx && g->feat_local_size && g->level_scale, "grid buffer is null");
	a.n_levels = g->n_levels;
	a.n_volumes = g->n_volumes;
	a.min_x = g->box_min[0]; a.min_y = g->box_min[1]; a.min_z = g->box_min[2];
	a.max_x = g->box_max[0]; a.max_y = g->box_max[1]; a.max_z = g->box_max[2];
	a.primes = g->primes;
	a.biases = g->biases;
	a.feat_local_idx = g->feat_local_idx;
	a.feat_local_size = g->feat_local_size;
	a.level_scale = g->level_scale;
	return NRF_OK;
}

// One work item per thread, 128-thread CTAs.  MEASURED AND NOT KEPT (gpurun_out/r2a/hash_plan_ab.jsonl -> profiles/r2_hash_plan_ab.jsonl): a
// one-wave persistent grid in which every SM gets the same number of items (k items per thread at a stride of the grid).  The coarse
// pass costs 1.75x the fine pass per point (95 us / 262 144 points vs 167 us / 786 432) and round 1 suspected the 15 %-full second
// wave of its launch; the balanced grid did not move it (97.6 us) and made the other launches slower (fine 166.6 -> 183.8 us, backward
// 264 -> 293 us).  The coarse pass is slower per point because its samples are 3x further apart along the ray: neighbouring lanes share
// a cell on fewer levels, so the warp's gathers coalesce into more distinct 32-byte sectors per point — the same L1-miss sector
// ceiling as the fine pass (1 sector / clk / SM), not a launch-shape effect.
struct LaunchPlan { unsigned grid; int64_t stride; int iters; };

static LaunchPlan launch_plan(int64_t items, int block)
{
	const int64_t ctas = (items + block - 1) / block;
	return {static_cast<unsigned>(ctas), ctas * block, 1};
}

}  // namespace nrf

using namespace nrf;

extern "C" {

int nrf_hash_level_scales(int32_t base_resolution, int32_t finest_resolution, int32_t n_levels, float* level_scale, nrf_stream stream)
{
	NRF_REQUIRE(level_scale != nullptr, "level_scale is null");
	NRF_REQUIRE(n_levels >= 1 && n_levels <= NRF_MAX_LEVELS, "n_levels out of range");
	level_scale_kernel<<<1, NRF_MAX_LEVELS, 0, as_stream(stream)>>>(base_resolution, finest_resolution, n_levels, level_scale);
	NRF_CHECK_LAUNCH("level_scale_kernel");
	return NRF_OK;
}

int nrf_hash_cells(const nrf_hash_grid* grid, const float* points, int64_t n_points, int clamp_points, int64_t* addr, float* weights,
	nrf_stream stream)
{
	HashArgs a;
	if (int rc = fill_args(grid, a)) return rc;
	NRF_REQUIRE(n_points >= 0, "negative n_points");
	if (n_points == 0) return NRF_OK;
	NRF_REQUIRE(points && addr && weights, "null pointer");
	hash_cells_kernel<<<static_cast<unsigned>((n_points + 127) / 128), 128, 0, as_stream(stream)>>>(a, points, n_points, clamp_points, grid->n_features,
		addr, weights);
	NRF_CHECK_LAUNCH("hash_cells_kernel");
	return NRF_OK;
}

int nrf_table_to_half(const float* table_f32, void* table_f16, int64_t n_scalars, nrf_stream stream)
{
	NRF_REQUIRE(table_f32 && table_f16, "null table");
	if (n_scalars <= 0) return NRF_OK;
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(table_f32) & 15) == 0 && (reinterpret_cast<uintptr_t>(table_f16) & 7) == 0, "tables must be 16-byte aligned");
	const int64_t quads = (n_scalars + 3) / 4;
	const int blocks = static_cast<int>(std::min<int64_t>((quads + 255) / 256, kNumSMs * 8));
	table_to_half_kernel<<<blocks, 256, 0, as_stream(stream)>>>(table_f32, reinterpret_cast<__half*>(table_f16), n_scalars);
	NRF_CHECK_LAUNCH("table_to_half_kernel");
	return NRF_OK;
}

}  // extern "C"

template <class PS>
static int launch_hash_fwd(const nrf_hash_grid* grid, const void* table_f16, const PS& ps, const Reuse& ru, int64_t n_points,
	int clamp_points, uint8_t* keep, void* enc_out, nrf_enc_layout layout, nrf_stream stream)
{
	HashArgs a;
	if (int rc = fill_args(grid, a)) return rc;
	NRF_REQUIRE(table_f16 && enc_out, "null table / output");
	NRF_REQUIRE(layout == NRF_ENC_F32 || layout == NRF_ENC_F16, "bad layout");
	const int F = grid->n_features;
	const __half* t = reinterpret_cast<const __half*>(table_f16);
	cudaStream_t s = as_stream(stream);
	// lanes per point: one per 16-byte chunk of the row at 16 levels (4 at F2, 8 at F4, 16 at F8); every other shape, for example L12 F2 or
	// L8 F8, runs one thread per point
	const int chunks = (grid->n_levels * F + 7) / 8;
	const bool split = (grid->n_levels * F) % 8 == 0 && (chunks & (chunks - 1)) == 0 && chunks <= 32 && chunks > 1;
#define NRF_LAUNCH_FWD2(FF, O32, SP)                                                                                              \
	do {                                                                                                                          \
		const int64_t items = (ps.group > 1 ? (static_cast<int64_t>(ps.R) + ps.group - 1) / ps.group * ps.group * ps.S_work : n_points) * (SP); \
		const LaunchPlan lp = launch_plan(items, 128);                                                                           \
		fwd_kernel<FF, O32, SP>(ps)<<<lp.grid, 128, 0, s>>>(a, t, ps, ru, items, lp.stride, lp.iters, clamp_points, keep, enc_out);       \
	} while (0)
#define NRF_LAUNCH_FWD(FF, SP)                                                     \
	do {                                                                           \
		if (layout == NRF_ENC_F32) NRF_LAUNCH_FWD2(FF, true, SP);                  \
		else NRF_LAUNCH_FWD2(FF, false, SP);                                       \
	} while (0)
	if (F == 2) { if (split && chunks == 4) NRF_LAUNCH_FWD(2, 4); else NRF_LAUNCH_FWD(2, 1); }
	else if (F == 4) { if (split && chunks == 8) NRF_LAUNCH_FWD(4, 8); else NRF_LAUNCH_FWD(4, 1); }
	else if (F == 8) { if (split && chunks == 16) NRF_LAUNCH_FWD(8, 16); else NRF_LAUNCH_FWD(8, 1); }
	else { set_error("nrf_hash_encode_fwd: n_features must be 2, 4 or 8"); return NRF_ERR_UNSUPPORTED; }
#undef NRF_LAUNCH_FWD
#undef NRF_LAUNCH_FWD2
	NRF_CHECK_LAUNCH("hash_fwd_kernel");
	return NRF_OK;
}

template <class PS>
static int launch_hash_bwd(const nrf_hash_grid* grid, const PS& ps, int64_t n_points, int clamp_points, const void* grad_enc,
	nrf_grad_layout layout, float* grad_table, nrf_stream stream)
{
	HashArgs a;
	if (int rc = fill_args(grid, a)) return rc;
	NRF_REQUIRE(grad_table != nullptr && grad_enc != nullptr, "null grad_table / grad");
	NRF_REQUIRE(layout == NRF_GRAD_F32 || layout == NRF_GRAD_BF16, "bad layout");
	const int F = grid->n_features;
	NRF_REQUIRE(F == 2 || F == 4 || F == 8, "n_features must be 2, 4 or 8");
	cudaStream_t s = as_stream(stream);
#define NRF_LAUNCH_BWD2(FF, BF)                                                                                                   \
	do {                                                                                                                          \
		const LaunchPlan lp = launch_plan(n_points, 128);                                                                        \
		bwd_kernel<FF, BF>(ps)<<<lp.grid, 128, 0, s>>>(a, ps, n_points, lp.stride, lp.iters, clamp_points, grad_enc, grad_table); \
	} while (0)
#define NRF_LAUNCH_BWD(FF)                                             \
	do {                                                               \
		if (layout == NRF_GRAD_BF16) NRF_LAUNCH_BWD2(FF, true);        \
		else NRF_LAUNCH_BWD2(FF, false);                               \
	} while (0)
	if (F == 2) { NRF_LAUNCH_BWD(2); }
	else if (F == 4) { NRF_LAUNCH_BWD(4); }
	else if (F == 8) { NRF_LAUNCH_BWD(8); }
	else { set_error("nrf_hash_encode_bwd: n_features must be 2, 4 or 8"); return NRF_ERR_UNSUPPORTED; }
#undef NRF_LAUNCH_BWD
#undef NRF_LAUNCH_BWD2
	NRF_CHECK_LAUNCH("hash_bwd_kernel");
	return NRF_OK;
}

extern "C" {

int nrf_hash_encode_fwd(const nrf_hash_grid* grid, const void* table_f16, const float* points, int64_t n_points,
	int clamp_points, uint8_t* keep, void* enc_out, nrf_enc_layout layout, nrf_stream stream)
{
	NRF_REQUIRE(n_points >= 0, "negative n_points");
	if (n_points == 0) { HashArgs a; return fill_args(grid, a); }
	NRF_REQUIRE(points != nullptr, "null points");
	const PointSrc ps{points, nullptr, nullptr, 0, 1};
	const Reuse ru{nullptr, nullptr, nullptr, 0};
	return launch_hash_fwd(grid, table_f16, ps, ru, n_points, clamp_points, keep, enc_out, layout, stream);
}

int nrf_hash_encode_bwd(const nrf_hash_grid* grid, const float* points, int64_t n_points, int clamp_points,
	const void* grad_enc, nrf_grad_layout layout, float* grad_table, nrf_stream stream)
{
	NRF_REQUIRE(n_points >= 0, "negative n_points");
	if (n_points == 0) { HashArgs a; return fill_args(grid, a); }
	NRF_REQUIRE(points != nullptr, "null points");
	const PointSrc ps{points, nullptr, nullptr, 0, 1};
	return launch_hash_bwd(grid, ps, n_points, clamp_points, grad_enc, layout, grad_table, stream);
}

int nrf_hash_encode_rays_fwd(const nrf_hash_grid* grid, const void* table_f16, const float* ray_batch, int32_t ray_stride, const float* z,
	int64_t n_rays, int32_t n_samples, int clamp_points, uint8_t* keep, void* enc_out, nrf_enc_layout layout, const int16_t* reuse_perm,
	const void* reuse_enc, const uint8_t* reuse_keep, int32_t reuse_samples, nrf_stream stream)
{
	return nrf_hash_encode_rays_fwd_grouped(grid, table_f16, ray_batch, ray_stride, z, n_rays, n_samples, clamp_points, keep, enc_out, layout, reuse_perm,
		reuse_enc, reuse_keep, reuse_samples, 1, stream);
}

int nrf_hash_encode_rays_fwd_grouped(const nrf_hash_grid* grid, const void* table_f16, const float* ray_batch, int32_t ray_stride, const float* z,
	int64_t n_rays, int32_t n_samples, int clamp_points, uint8_t* keep, void* enc_out, nrf_enc_layout layout, const int16_t* reuse_perm,
	const void* reuse_enc, const uint8_t* reuse_keep, int32_t reuse_samples, int32_t ray_group, nrf_stream stream)
{
	NRF_REQUIRE(ray_group >= 1 && ray_group <= 1024, "ray_group out of range");
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1 && ray_stride >= 6, "bad sizes");
	if (n_rays == 0) { HashArgs a; return fill_args(grid, a); }
	NRF_REQUIRE(ray_batch && z, "null ray_batch / z");
	const int64_t n_points = n_rays * n_samples;
	NRF_REQUIRE(n_points < (int64_t(1) << 31), "n_rays * n_samples must be < 2^31 per call");
	Reuse ru{nullptr, nullptr, nullptr, 0};
	if (reuse_perm) {
		NRF_REQUIRE(grid != nullptr && reuse_samples >= 1 && reuse_samples <= n_samples && n_samples < 32768, "bad reuse arguments");
		const int row_bytes = grid->n_levels * grid->n_features * (layout == NRF_ENC_F32 ? 4 : 2);
		NRF_REQUIRE(row_bytes % 16 == 0 && ((reinterpret_cast<uintptr_t>(reuse_enc) | reinterpret_cast<uintptr_t>(enc_out)) & 15) == 0,
			"row reuse needs 16-byte aligned rows");
		ru = Reuse{reuse_perm, reuse_enc, reuse_keep, reuse_samples};
	}
	NRF_REQUIRE((n_rays + ray_group) * n_samples < (int64_t(1) << 31), "(n_rays + ray_group) * n_samples must be < 2^31 per call");
	const int s_work = reuse_perm && !reuse_enc && ray_group > 1 ? n_samples - reuse_samples : n_samples;   // nothing to copy: skip those items
	const PointSrc ps{nullptr, ray_batch, z, ray_stride, n_samples, ray_group, static_cast<int>(n_rays), s_work};
	return launch_hash_fwd(grid, table_f16, ps, ru, n_points, clamp_points, keep, enc_out, layout, stream);
}

int nrf_hash_encode_rays_bwd(const nrf_hash_grid* grid, const float* ray_batch, int32_t ray_stride, const float* z, int64_t n_rays,
	int32_t n_samples, int clamp_points, const void* grad_enc, nrf_grad_layout layout, float* grad_table, nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1 && ray_stride >= 6, "bad sizes");
	if (n_rays == 0) { HashArgs a; return fill_args(grid, a); }
	NRF_REQUIRE(ray_batch && z, "null ray_batch / z");
	const int64_t n_points = n_rays * n_samples;
	NRF_REQUIRE(n_points < (int64_t(1) << 31), "n_rays * n_samples must be < 2^31 per call");
	const PointSrc ps{nullptr, ray_batch, z, ray_stride, n_samples};
	return launch_hash_bwd(grid, ps, n_points, clamp_points, grad_enc, layout, grad_table, stream);
}


// argument checks and the point source of the two jitter entries
static int jitter_src(const nrf_hash_grid* grid, const float* ray_batch, int32_t ray_stride, const float* z, int64_t n_rays, int32_t n_samples,
	const nrf_point_jitter* j, JitterSrc& ps)
{
	NRF_REQUIRE(grid != nullptr && j != nullptr, "null grid / jitter");
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1 && ray_stride >= 6, "bad sizes");
	NRF_REQUIRE(n_rays * n_samples < (int64_t(1) << 31), "n_rays * n_samples must be < 2^31 per call");
	NRF_REQUIRE(!j->cone_angle || (j->rand_r && j->rand_theta && j->cone_stride >= 0), "a cone needs rand_r, rand_theta and cone_stride >= 0");
	NRF_REQUIRE(!j->sp_noise || j->sp_alpha, "sp_noise needs the device scalar sp_alpha");
	NRF_REQUIRE(n_rays == 0 || (ray_batch && z), "null ray_batch / z");
	ps = JitterSrc{ray_batch, z, ray_stride, n_samples, j->cone_angle, j->cone_stride, j->rand_r, j->rand_theta, j->clamp_to_box, j->sp_noise, j->sp_alpha, {}};
	for (int k = 0; k < 3; k++) { ps.box.lo[k] = grid->box_min[k]; ps.box.hi[k] = grid->box_max[k]; }
	return NRF_OK;
}

int nrf_hash_encode_rays_jitter_fwd(const nrf_hash_grid* grid, const void* table_f16, const float* ray_batch, int32_t ray_stride, const float* z,
	int64_t n_rays, int32_t n_samples, int clamp_points, uint8_t* keep, void* enc_out, nrf_enc_layout layout, const nrf_point_jitter* jitter,
	nrf_stream stream)
{
	JitterSrc ps;
	if (int rc = jitter_src(grid, ray_batch, ray_stride, z, n_rays, n_samples, jitter, ps)) return rc;
	if (n_rays == 0) { HashArgs a; return fill_args(grid, a); }
	const Reuse ru{nullptr, nullptr, nullptr, 0};
	return launch_hash_fwd(grid, table_f16, ps, ru, n_rays * n_samples, clamp_points, keep, enc_out, layout, stream);
}

int nrf_hash_encode_rays_jitter_bwd(const nrf_hash_grid* grid, const float* ray_batch, int32_t ray_stride, const float* z, int64_t n_rays,
	int32_t n_samples, int clamp_points, const void* grad_enc, nrf_grad_layout layout, float* grad_table, const nrf_point_jitter* jitter,
	nrf_stream stream)
{
	JitterSrc ps;
	if (int rc = jitter_src(grid, ray_batch, ray_stride, z, n_rays, n_samples, jitter, ps)) return rc;
	if (n_rays == 0) { HashArgs a; return fill_args(grid, a); }
	return launch_hash_bwd(grid, ps, n_rays * n_samples, clamp_points, grad_enc, layout, grad_table, stream);
}

}
