// Ray generation, AABB clipping, depth sampling and point generation for sm_100a.
//
// Replaces the ~40 tiny ATen launches of GetRays / IntersectWithAABB (reference src/RayUtils.h:5-46, 87-126), the
// Render prologue (src/NeRFRenderer.h:549-583) and the z / point construction of RenderRays (:384-419, :432).
// Arithmetic keeps ATen's un-fused order (__fmul_rn / __fadd_rn, no FMA contraction) so that z values, and through
// them the sample points and hash cells, are the same floats the reference produces.
#include "common.cuh"
#include "jitter.cuh"
#include "sh_basis.cuh"

namespace nrf {

struct Cam {
	float fx, fy, cx, cy;
	float m[12];  // c2w[:3,:4] row-major
};

// GetDirections + the rotation into the world frame for ONE pixel (src/RayUtils.h:5-32; NeRFDataset::GetRayBatch, src/NeRFDataset.cpp:117-131,
// is the same expression on a list of pixel coordinates)
__device__ __forceinline__ void pixel_ray(const Cam& c, int py, int px, float (&o)[3], float (&d)[3])
{
	const float dx = __fdiv_rn(__fsub_rn(static_cast<float>(px), c.cx), c.fx);
	const float dy = -__fdiv_rn(__fsub_rn(static_cast<float>(py), c.cy), c.fy);
	const float dz = -1.f;
#pragma unroll
	for (int r = 0; r < 3; r++) {
		d[r] = __fadd_rn(__fadd_rn(__fmul_rn(dx, c.m[r * 4 + 0]), __fmul_rn(dy, c.m[r * 4 + 1])), __fmul_rn(dz, c.m[r * 4 + 2]));
		o[r] = c.m[r * 4 + 3];
	}
}

__global__ void __launch_bounds__(256) get_rays_kernel(Cam c, int w, int row_begin, int64_t n, float* __restrict__ rays_o, float* __restrict__ rays_d)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const int py = row_begin + static_cast<int>(i / w), px = static_cast<int>(i % w);
	// GetDirections (src/RayUtils.h:5-21), rays_d = sum(dirs[..., None, :] * c2w[:3,:3], -1) (:28-32)
	float o[3], d[3];
	pixel_ray(c, py, px, o, d);
#pragma unroll
	for (int r = 0; r < 3; r++) { rays_d[i * 3 + r] = d[r]; rays_o[i * 3 + r] = o[r]; }
}

// NeRFDataset::GetRayBatch (src/NeRFDataset.cpp:109-144) and the target gather of get_batch (:156: CurrentImage.index({rand_h, rand_w}))
__global__ void __launch_bounds__(256) ray_batch_kernel(Cam c, const int32_t* __restrict__ pix_hw, int64_t n, const float* __restrict__ image, int img_w, int img_c,
	float* __restrict__ rays_o, float* __restrict__ rays_d, float* __restrict__ target)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const int py = pix_hw[2 * i], px = pix_hw[2 * i + 1];
	float o[3], d[3];
	pixel_ray(c, py, px, o, d);
#pragma unroll
	for (int r = 0; r < 3; r++) { rays_o[i * 3 + r] = o[r]; rays_d[i * 3 + r] = d[r]; }
	if (image && target) {
		const float* src = image + (static_cast<int64_t>(py) * img_w + px) * img_c;
		for (int k = 0; k < img_c; k++) target[i * img_c + k] = __ldg(src + k);
	}
}

// IntersectWithAABB (src/RayUtils.h:87-126) and viewdirs = rays_d / norm(rays_d) (src/NeRFRenderer.h:559) for one ray
__device__ __forceinline__ void prepare_ray(const float (&o)[3], const float (&d)[3], const Box& box, float near_plane, float& tnear, float& tfar,
	float (&vd)[3])
{
	tnear = -INFINITY;
	tfar = INFINITY;
#pragma unroll
	for (int k = 0; k < 3; k++) {
		const float frac = __fdiv_rn(1.0f, __fadd_rn(d[k], 1e-6f));
		const float t1 = __fmul_rn(__fsub_rn(box.lo[k], o[k]), frac);
		const float t2 = __fmul_rn(__fsub_rn(box.hi[k], o[k]), frac);
		tnear = fmaxf(tnear, fminf(t1, t2));
		tfar = fminf(tfar, fmaxf(t1, t2));
	}
	tnear = fmaxf(tnear, near_plane);
	tfar = fmaxf(tfar, __fadd_rn(tnear, 1e-6f));
	const float nrm = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(d[0], d[0]), __fmul_rn(d[1], d[1])), __fmul_rn(d[2], d[2])));
#pragma unroll
	for (int k = 0; k < 3; k++) vd[k] = __fdiv_rn(d[k], nrm);
}

__global__ void __launch_bounds__(256) rays_prepare_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d,
	int64_t n, Box box, float near_plane, int use_viewdirs, float* __restrict__ ray_batch)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) return;
	float o[3], d[3], vd[3], tnear, tfar;
#pragma unroll
	for (int k = 0; k < 3; k++) { o[k] = rays_o[i * 3 + k]; d[k] = rays_d[i * 3 + k]; }
	prepare_ray(o, d, box, near_plane, tnear, tfar, vd);
	const int stride = use_viewdirs ? 11 : 8;
	float* out = ray_batch + i * stride;
#pragma unroll
	for (int k = 0; k < 3; k++) { out[k] = o[k]; out[3 + k] = d[k]; }
	out[6] = tnear;
	out[7] = tfar;
	if (use_viewdirs) {
#pragma unroll
		for (int k = 0; k < 3; k++) out[8 + k] = vd[k];
	}
}

__device__ __forceinline__ float safe_inv(float x) { return fabsf(x) < 1e-8f ? __fdiv_rn(1.0f, 1e-8f) : __fdiv_rn(1.0f, x); }

// z = near (1 - t) + far t, or its lin_disp form (src/NeRFRenderer.h:397, :400-401)
__device__ __forceinline__ float z_value(float nr, float fr, float t, int lin_disp)
{
	const float omt = __fsub_rn(1.f, t);
	if (!lin_disp) return __fadd_rn(__fmul_rn(nr, omt), __fmul_rn(fr, t));
	return safe_inv(__fadd_rn(__fmul_rn(safe_inv(nr), omt), __fmul_rn(safe_inv(fr), t)));
}

__global__ void __launch_bounds__(256) z_sample_kernel(const float* __restrict__ ray_batch, int ray_stride, const float* __restrict__ t_vals,
	int64_t R, int S, int lin_disp, float* __restrict__ z)
{
	const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (e >= R * S) return;
	const int64_t ray = e / S;
	const int s = static_cast<int>(e % S);
	z[e] = z_value(ray_batch[ray * ray_stride + 6], ray_batch[ray * ray_stride + 7], t_vals[s], lin_disp);
}

// Render prologue + coarse depths + per-ray SH table in ONE launch (the head of every RenderRays call: three kernels and, in a training
// step, the memset of the loss accumulator).  One thread per (ray, sample): each recomputes its ray's slab test (a dozen flops, the same
// operations in the same order, hence the same near / far) and writes its z; the thread of sample 0 also writes the ray's [o, d, near,
// far, viewdirs] row and its SH basis.  Bit-identical to nrf_rays_prepare + nrf_z_sample + nrf_sh_encode_fwd.
// PIXELS: the rays come from pixel coordinates + the camera (ray_batch_kernel's arithmetic) instead of rays_o / rays_d arrays, which are then
// OUTPUTS (the compositing kernels read rays_d), as is the gathered target.
struct PixelSrc {
	Cam cam;
	const int32_t* pix_hw;     // [R,2] (row, column), or nullptr: ray r is pixel first_pixel + r of the image in GetRays order (row-major, img_w wide)
	int64_t first_pixel;
	const float* image;
	int img_w, img_c;
	float* rays_o_out;
	float* rays_d_out;
	float* target_out;
	// or: the rays arrive as rows [o(3) d(3) near far viewdirs(3)] of an already prepared batch (what BatchifyRays hands to RenderRays,
	// src/NeRFRenderer.h:483): near / far / viewdirs are TAKEN from it, not recomputed
	const float* prepared;
	int prepared_stride;
};

template <int DEG, bool PIXELS>
__global__ void __launch_bounds__(256) ray_setup_kernel(const float* __restrict__ rays_o, const float* __restrict__ rays_d, PixelSrc ps, int64_t R, Box box,
	float near_plane, const float* __restrict__ t_vals, int S, int lin_disp, float* __restrict__ ray_batch, float* __restrict__ z,
	float* __restrict__ ray_sh, float* __restrict__ zero_scalar)
{
	const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (e == 0 && zero_scalar) *zero_scalar = 0.f;
	if (e >= R * S) return;
	const int64_t ray = e / S;
	const int s = static_cast<int>(e % S);
	float o[3], d[3], vd[3], tnear, tfar;
	bool prepared = false;
	if (PIXELS) {
		if (ps.prepared) {
			const float* rb = ps.prepared + ray * ps.prepared_stride;
#pragma unroll
			for (int k = 0; k < 3; k++) { o[k] = rb[k]; d[k] = rb[3 + k]; vd[k] = rb[8 + k]; }
			tnear = rb[6];
			tfar = rb[7];
			prepared = true;
		} else {
			int py, px;
			if (ps.pix_hw) {
				py = ps.pix_hw[2 * ray];
				px = ps.pix_hw[2 * ray + 1];
			} else {
				const int64_t lin = ps.first_pixel + ray;
				py = static_cast<int>(lin / ps.img_w);
				px = static_cast<int>(lin - static_cast<int64_t>(py) * ps.img_w);
			}
			pixel_ray(ps.cam, py, px, o, d);
			if (s == 0 && ps.image && ps.target_out) {
				const float* src = ps.image + (static_cast<int64_t>(py) * ps.img_w + px) * ps.img_c;
				for (int k = 0; k < ps.img_c; k++) ps.target_out[ray * ps.img_c + k] = __ldg(src + k);
			}
		}
		if (s == 0) {
#pragma unroll
			for (int k = 0; k < 3; k++) {
				if (ps.rays_o_out) ps.rays_o_out[ray * 3 + k] = o[k];
				ps.rays_d_out[ray * 3 + k] = d[k];
			}
		}
	} else {
#pragma unroll
		for (int k = 0; k < 3; k++) { o[k] = rays_o[ray * 3 + k]; d[k] = rays_d[ray * 3 + k]; }
	}
	if (!prepared) prepare_ray(o, d, box, near_plane, tnear, tfar, vd);
	z[e] = z_value(tnear, tfar, t_vals[s], lin_disp);
	if (s == 0) {
		float* out = ray_batch + ray * 11;
#pragma unroll
		for (int k = 0; k < 3; k++) { out[k] = o[k]; out[3 + k] = d[k]; out[8 + k] = vd[k]; }
		out[6] = tnear;
		out[7] = tfar;
		if (ray_sh) {
			float b[DEG * DEG];
			sh_basis<DEG>(vd[0], vd[1], vd[2], b);
#pragma unroll
			for (int k = 0; k < DEG * DEG; k++) ray_sh[ray * (DEG * DEG) + k] = b[k];
		}
	}
}

__global__ void __launch_bounds__(256) sample_points_kernel(const float* __restrict__ ray_batch, int ray_stride, const float* __restrict__ z,
	int64_t R, int S, float* __restrict__ pts)
{
	// one thread per output scalar: stores are contiguous
	const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (e >= R * S * 3) return;
	const int64_t smp = e / 3;
	const int k = static_cast<int>(e % 3);
	const int64_t ray = smp / S;
	const float* rb = ray_batch + ray * ray_stride;
	pts[e] = __fadd_rn(rb[k], __fmul_rn(rb[3 + k], z[smp]));  // src/NeRFRenderer.h:419
}

// TangentScatter (src/NeRFRenderer.h:307-362): in-cone jitter of the sample points.  The two uniform variates per sample are
// INPUTS (the host draws them with the same two torch::rand calls as the reference, :342-343, so the Philox stream stays
// in lock-step with it); this kernel fuses the ~40 ATen launches that build the tangent frame and apply the offset (jitter.cuh).
__global__ void __launch_bounds__(256) tangent_scatter_kernel(float* __restrict__ pts, const float* __restrict__ z,
	const float* __restrict__ cone_angle, int cone_stride, const float* __restrict__ rays_d, int d_stride,
	const float* __restrict__ rand_r, const float* __restrict__ rand_theta, Box box, int clamp_box, int64_t R, int S)
{
	const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (e >= R * S) return;
	const int64_t ray = e / S;
	float off[3];
	tangent_direction(rays_d[ray * d_stride], rays_d[ray * d_stride + 1], rays_d[ray * d_stride + 2], rand_r[e], rand_theta[e], off);
	const float radius = __fmul_rn(cone_angle[cone_stride ? ray * cone_stride : 0], z[e]);   // cone_radii = cone_angle * z (:313)
	float* p = pts + e * 3;
	float px = p[0], py = p[1], pz = p[2];
	apply_tangent_offset(off, radius, px, py, pz);
	if (clamp_box) clamp_to_box(box, px, py, pz);
	p[0] = px; p[1] = py; p[2] = pz;
}

// Stochastic preconditioning of the fine-pass sample positions (src/NeRFRenderer.h:435-443) + ReflectBoundary (:285-304), jitter.cuh.  noise
// [R,S,3] standard normal (the reference's torch::randn_like draw, supplied by the host so that the Philox stream is the caller's).
__global__ void __launch_bounds__(256) precondition_kernel(float* __restrict__ pts, const float* __restrict__ noise, float alpha, Box box, int64_t n3)
{
	const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (e >= n3) return;
	const int k = static_cast<int>(e % 3);
	pts[e] = precondition_coord(pts[e], noise[e], alpha, box.lo[k], box.hi[k]);
}

}  // namespace nrf

using namespace nrf;

static void fill_cam(Cam& c, const float* K_host, const float* c2w_host)
{
	c.fx = K_host[0]; c.cx = K_host[2]; c.fy = K_host[4]; c.cy = K_host[5];
	for (int i = 0; i < 12; i++) c.m[i] = c2w_host[i];
}

extern "C" {

int nrf_get_rays(int32_t h, int32_t w, const float* K_host, const float* c2w_host, int32_t row_begin, int32_t row_end,
	float* rays_o, float* rays_d, nrf_stream stream)
{
	NRF_REQUIRE(h > 0 && w > 0 && row_begin >= 0 && row_end <= h && row_begin <= row_end, "bad image / tile size");
	NRF_REQUIRE(K_host && c2w_host, "null camera");
	const int64_t n = static_cast<int64_t>(row_end - row_begin) * w;
	if (n == 0) return NRF_OK;
	NRF_REQUIRE(rays_o && rays_d, "null output");
	Cam c;
	fill_cam(c, K_host, c2w_host);
	get_rays_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, as_stream(stream)>>>(c, w, row_begin, n, rays_o, rays_d);
	NRF_CHECK_LAUNCH("get_rays_kernel");
	return NRF_OK;
}

int nrf_rays_prepare(const float* rays_o, const float* rays_d, int64_t n_rays, const float* bbox_host, float near_plane,
	int32_t use_viewdirs, float* ray_batch, nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0, "bad sizes");
	NRF_REQUIRE(bbox_host != nullptr, "null bbox");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(rays_o && rays_d && ray_batch, "null pointer");
	Box b;
	for (int k = 0; k < 3; k++) { b.lo[k] = bbox_host[k]; b.hi[k] = bbox_host[3 + k]; }
	rays_prepare_kernel<<<static_cast<unsigned>((n_rays + 255) / 256), 256, 0, as_stream(stream)>>>(rays_o, rays_d, n_rays, b, near_plane, use_viewdirs, ray_batch);
	NRF_CHECK_LAUNCH("rays_prepare_kernel");
	return NRF_OK;
}

int nrf_ray_batch(const int32_t* pix_hw, int64_t n_rays, const float* K_host, const float* c2w_host, const float* image, int32_t img_h, int32_t img_w,
	int32_t img_c, float* rays_o, float* rays_d, float* target, float* cone_angle_host, nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0, "bad sizes");
	NRF_REQUIRE(K_host && c2w_host, "null camera");
	if (cone_angle_host) *cone_angle_host = (1.0f / K_host[0] + 1.0f / K_host[4]) / 2.0f;      // src/NeRFDataset.cpp:136-141
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(pix_hw && rays_o && rays_d, "null pointer");
	NRF_REQUIRE((image == nullptr) == (target == nullptr) && (!image || (img_h > 0 && img_w > 0 && img_c > 0)), "image and target go together");
	Cam c;
	fill_cam(c, K_host, c2w_host);
	ray_batch_kernel<<<static_cast<unsigned>((n_rays + 255) / 256), 256, 0, as_stream(stream)>>>(c, pix_hw, n_rays, image, img_w, img_c, rays_o, rays_d, target);
	NRF_CHECK_LAUNCH("ray_batch_kernel");
	return NRF_OK;
}

static int launch_ray_setup(bool pixels, const float* rays_o, const float* rays_d, const PixelSrc& ps, int64_t n_rays, const float* bbox_host, float near_plane,
	const float* t_vals, int32_t n_samples, int32_t lin_disp, int32_t sh_degree, float* ray_batch, float* z, float* ray_sh, float* zero_scalar, nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1, "bad sizes");
	NRF_REQUIRE(!ray_sh || (sh_degree >= 1 && sh_degree <= 8), "degree must be 1..8");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(bbox_host && t_vals && ray_batch && z, "null pointer");
	Box b;
	for (int k = 0; k < 3; k++) { b.lo[k] = bbox_host[k]; b.hi[k] = bbox_host[3 + k]; }
	const int64_t n = n_rays * n_samples;
	const unsigned blocks = static_cast<unsigned>((n + 255) / 256);
	cudaStream_t s = as_stream(stream);
#define NRF_RS(D) case D:                                                                                                                                     \
		if (pixels) ray_setup_kernel<D, true><<<blocks, 256, 0, s>>>(rays_o, rays_d, ps, n_rays, b, near_plane, t_vals, n_samples, lin_disp, ray_batch, z, ray_sh, zero_scalar); \
		else ray_setup_kernel<D, false><<<blocks, 256, 0, s>>>(rays_o, rays_d, ps, n_rays, b, near_plane, t_vals, n_samples, lin_disp, ray_batch, z, ray_sh, zero_scalar);   \
		break
	switch (ray_sh ? sh_degree : 1) {
		NRF_RS(1); NRF_RS(2); NRF_RS(3); NRF_RS(4); NRF_RS(5); NRF_RS(6); NRF_RS(7); NRF_RS(8);
	}
#undef NRF_RS
	NRF_CHECK_LAUNCH("ray_setup_kernel");
	return NRF_OK;
}

int nrf_ray_setup(const float* rays_o, const float* rays_d, int64_t n_rays, const float* bbox_host, float near_plane, const float* t_vals,
	int32_t n_samples, int32_t lin_disp, int32_t sh_degree, float* ray_batch, float* z, float* ray_sh, float* zero_scalar, nrf_stream stream)
{
	NRF_REQUIRE(n_rays <= 0 || (rays_o && rays_d), "null pointer");
	const PixelSrc ps{};
	return launch_ray_setup(false, rays_o, rays_d, ps, n_rays, bbox_host, near_plane, t_vals, n_samples, lin_disp, sh_degree, ray_batch, z, ray_sh, zero_scalar, stream);
}

int nrf_ray_setup_pixels(const int32_t* pix_hw, int64_t n_rays, const float* K_host, const float* c2w_host, const float* image, int32_t img_h, int32_t img_w,
	int32_t img_c, const float* bbox_host, float near_plane, const float* t_vals, int32_t n_samples, int32_t lin_disp, int32_t sh_degree, float* rays_o,
	float* rays_d, float* target, float* ray_batch, float* z, float* ray_sh, float* zero_scalar, nrf_stream stream)
{
	NRF_REQUIRE(K_host && c2w_host, "null camera");
	NRF_REQUIRE(n_rays <= 0 || (pix_hw && rays_o && rays_d), "null pointer");
	NRF_REQUIRE((image == nullptr) == (target == nullptr) && (!image || (img_h > 0 && img_w > 0 && img_c > 0)), "image and target go together");
	PixelSrc ps{};
	fill_cam(ps.cam, K_host, c2w_host);
	ps.pix_hw = pix_hw; ps.image = image; ps.img_w = img_w; ps.img_c = img_c; ps.rays_o_out = rays_o; ps.rays_d_out = rays_d; ps.target_out = target;
	return launch_ray_setup(true, nullptr, nullptr, ps, n_rays, bbox_host, near_plane, t_vals, n_samples, lin_disp, sh_degree, ray_batch, z, ray_sh, zero_scalar, stream);
}

int nrf_ray_setup_tile(const float* K_host, const float* c2w_host, int32_t img_w, int64_t first_pixel, int64_t n_rays, const float* bbox_host, float near_plane,
	const float* t_vals, int32_t n_samples, int32_t lin_disp, int32_t sh_degree, float* rays_o, float* rays_d, float* ray_batch, float* z, float* ray_sh,
	nrf_stream stream)
{
	NRF_REQUIRE(K_host && c2w_host, "null camera");
	NRF_REQUIRE(img_w > 0 && first_pixel >= 0, "bad image width / first pixel");
	NRF_REQUIRE(n_rays <= 0 || rays_d, "null rays_d");
	PixelSrc ps{};
	fill_cam(ps.cam, K_host, c2w_host);
	ps.first_pixel = first_pixel; ps.img_w = img_w; ps.rays_o_out = rays_o; ps.rays_d_out = rays_d;
	return launch_ray_setup(true, nullptr, nullptr, ps, n_rays, bbox_host, near_plane, t_vals, n_samples, lin_disp, sh_degree, ray_batch, z, ray_sh, nullptr, stream);
}

int nrf_ray_setup_prepared(const float* ray_batch_in, int32_t ray_stride, int64_t n_rays, const float* t_vals, int32_t n_samples, int32_t lin_disp,
	int32_t sh_degree, float* rays_d, float* ray_batch, float* z, float* ray_sh, nrf_stream stream)
{
	NRF_REQUIRE(ray_stride >= 11, "a prepared ray batch has rows [o d near far viewdirs]: ray_stride >= 11");
	NRF_REQUIRE(n_rays <= 0 || (ray_batch_in && rays_d), "null pointer");
	PixelSrc ps{};
	ps.prepared = ray_batch_in; ps.prepared_stride = ray_stride; ps.rays_d_out = rays_d;
	const float no_box[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};     // never read: near / far come with the batch
	return launch_ray_setup(true, nullptr, nullptr, ps, n_rays, no_box, 0.f, t_vals, n_samples, lin_disp, sh_degree, ray_batch, z, ray_sh, nullptr, stream);
}

int nrf_z_sample(const float* ray_batch, int32_t ray_stride, const float* t_vals, int64_t n_rays, int32_t n_samples,
	int32_t lin_disp, float* z, nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1 && ray_stride >= 8, "bad sizes");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(ray_batch && t_vals && z, "null pointer");
	const int64_t n = n_rays * n_samples;
	z_sample_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, as_stream(stream)>>>(ray_batch, ray_stride, t_vals, n_rays, n_samples, lin_disp, z);
	NRF_CHECK_LAUNCH("z_sample_kernel");
	return NRF_OK;
}

int nrf_sample_points(const float* ray_batch, int32_t ray_stride, const float* z, int64_t n_rays, int32_t n_samples,
	float* pts, nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1 && ray_stride >= 8, "bad sizes");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(ray_batch && z && pts, "null pointer");
	const int64_t n = n_rays * n_samples * 3;
	sample_points_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, as_stream(stream)>>>(ray_batch, ray_stride, z, n_rays, n_samples, pts);
	NRF_CHECK_LAUNCH("sample_points_kernel");
	return NRF_OK;
}

int nrf_precondition_points(float* pts, const float* noise, float alpha, const float* bbox_host, int64_t n_points, nrf_stream stream)
{
	NRF_REQUIRE(n_points >= 0 && bbox_host != nullptr, "bad arguments");
	if (n_points == 0) return NRF_OK;
	NRF_REQUIRE(pts && noise, "null pointer");
	Box b;
	for (int k = 0; k < 3; k++) { b.lo[k] = bbox_host[k]; b.hi[k] = bbox_host[3 + k]; }
	const int64_t n3 = n_points * 3;
	precondition_kernel<<<static_cast<unsigned>((n3 + 255) / 256), 256, 0, as_stream(stream)>>>(pts, noise, alpha, b, n3);
	NRF_CHECK_LAUNCH("precondition_kernel");
	return NRF_OK;
}

int nrf_tangent_scatter(float* pts, const float* z, const float* cone_angle, int32_t cone_stride, const float* rays_d,
	int32_t dir_stride, const float* rand_r, const float* rand_theta, const float* bbox_host, int64_t n_rays, int32_t n_samples,
	nrf_stream stream)
{
	NRF_REQUIRE(n_rays >= 0 && n_samples >= 1 && dir_stride >= 3 && cone_stride >= 0, "bad sizes");
	if (n_rays == 0) return NRF_OK;
	NRF_REQUIRE(pts && z && cone_angle && rays_d && rand_r && rand_theta, "null pointer");
	Box b{};
	if (bbox_host) for (int k = 0; k < 3; k++) { b.lo[k] = bbox_host[k]; b.hi[k] = bbox_host[3 + k]; }
	const int64_t n = n_rays * n_samples;
	tangent_scatter_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, as_stream(stream)>>>(pts, z, cone_angle, cone_stride, rays_d,
		dir_stride, rand_r, rand_theta, b, bbox_host != nullptr, n_rays, n_samples);
	NRF_CHECK_LAUNCH("tangent_scatter_kernel");
	return NRF_OK;
}

}
