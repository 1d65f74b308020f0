// Per-sample perturbations of the reference's shipped training configuration, as device functions shared by the kernels that materialise
// the jittered points (rays.cu: tangent_scatter_kernel, precondition_kernel) and the hash encode kernels that generate them in-kernel
// (hash_encode.cu: nrf_hash_encode_rays_jitter_fwd / _bwd).  One body for both, so both produce the same bits by construction.
// Arithmetic keeps ATen's un-fused order (__f*_rn, no FMA contraction), as the reference's tensor expressions round.
#pragma once
#include "common.cuh"

namespace nrf {

struct Box {
	float lo[3], hi[3];
};

__device__ __forceinline__ void safe_normalize3(float& x, float& y, float& z)
{
	const float n = fmaxf(sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z))), 1e-8f);
	x = __fdiv_rn(x, n); y = __fdiv_rn(y, n); z = __fdiv_rn(z, n);
}

// TangentScatter (src/NeRFRenderer.h:307-362) for one sample: the in-disc direction t r cos(theta) + b r sin(theta), with (dx, dy, dz) the ray's
// direction and u_r / u_theta the sample's two torch::rand variates (:342-343).  apply_tangent_offset scales it by the cone radius.
__device__ __forceinline__ void tangent_direction(float dx, float dy, float dz, float u_r, float u_theta, float (&off)[3])
{
	safe_normalize3(dx, dy, dz);
	// helper axis: the coordinate axis along which |d| is strictly smallest, z otherwise (:321-331)
	const float ax = fabsf(dx), ay = fabsf(dy), az = fabsf(dz);
	float ux = 0.f, uy = 0.f, uz = 0.f;
	if (ax < ay && ax < az) ux = 1.f;
	else if (ay < ax && ay < az) uy = 1.f;
	else uz = 1.f;
	// tangent = normalize(d x up), bitangent = normalize(d x tangent) (:333-336)
	float tx = __fsub_rn(__fmul_rn(dy, uz), __fmul_rn(dz, uy));
	float ty = __fsub_rn(__fmul_rn(dz, ux), __fmul_rn(dx, uz));
	float tz = __fsub_rn(__fmul_rn(dx, uy), __fmul_rn(dy, ux));
	safe_normalize3(tx, ty, tz);
	float bx = __fsub_rn(__fmul_rn(dy, tz), __fmul_rn(dz, ty));
	float by = __fsub_rn(__fmul_rn(dz, tx), __fmul_rn(dx, tz));
	float bz = __fsub_rn(__fmul_rn(dx, ty), __fmul_rn(dy, tx));
	safe_normalize3(bx, by, bz);
	// uniform over the disc: r = sqrt(clamp(u1)), theta = fmod(u2 * 2 pi, 2 pi) (:342-345)
	const float r = sqrtf(fminf(fmaxf(u_r, 1e-8f), 1.0f - 1e-8f));
	const float two_pi = 6.283185307179586f;
	const float theta = fmodf(__fmul_rn(__fmul_rn(u_theta, 2.0f), 3.14159265358979323846f), two_pi);
	const float ox = __fmul_rn(r, cosf(theta)), oy = __fmul_rn(r, sinf(theta));
	off[0] = __fadd_rn(__fmul_rn(tx, ox), __fmul_rn(bx, oy));
	off[1] = __fadd_rn(__fmul_rn(ty, ox), __fmul_rn(by, oy));
	off[2] = __fadd_rn(__fmul_rn(tz, ox), __fmul_rn(bz, oy));
}

// p += offset * radius, radius = cone_angle * z (:313, :361)
__device__ __forceinline__ void apply_tangent_offset(const float (&off)[3], float radius, float& px, float& py, float& pz)
{
	px = __fadd_rn(px, __fmul_rn(off[0], radius));
	py = __fadd_rn(py, __fmul_rn(off[1], radius));
	pz = __fadd_rn(pz, __fmul_rn(off[2], radius));
}

// TangentScatter's clamp into the bounding box (:356-360)
__device__ __forceinline__ void clamp_to_box(const Box& box, float& px, float& py, float& pz)
{
	px = fminf(fmaxf(px, box.lo[0]), box.hi[0]);
	py = fminf(fmaxf(py, box.lo[1]), box.hi[1]);
	pz = fminf(fmaxf(pz, box.lo[2]), box.hi[2]);
}

// Stochastic preconditioning of one coordinate (src/NeRFRenderer.h:435-443): p + noise * alpha, then ReflectBoundary (:285-304): normalise to
// the box, fold with period 2 (fmod; q -> 2 - q above 1), map back.
__device__ __forceinline__ float precondition_coord(float p, float noise, float alpha, float lo, float hi)
{
	const float ext = __fsub_rn(hi, lo);
	const float s = __fadd_rn(p, __fmul_rn(noise, alpha));
	float q = fmodf(__fdiv_rn(__fsub_rn(s, lo), ext), 2.0f);
	q = q > 1.0f ? __fsub_rn(2.0f, q) : q;
	return __fadd_rn(__fmul_rn(q, ext), lo);
}

}  // namespace nrf
