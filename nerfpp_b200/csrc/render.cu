// nrf_render_rays_fwd: RenderRays for inference (reference src/NeRFRenderer.h:366-459 with the Render prologue :549-583) as
// ONE C-ABI call for the <CuHashEmbedder, CuSHEncoder, NeRFSmall> instantiation.
//
// Host-side sequencing only: it enqueues the kernels of this library on the caller's stream in the reference's order —
//   ray prologue (viewdirs, IntersectWithAABB) -> SH per ray -> z = near(1-t)+far t -> [hash encode (points generated in-kernel)
//   -> fused MLP (keep mask in the epilogue)] -> RawToOutputs -> SamplePDF + merge -> second network pass -> RawToOutputs
// — into a caller-owned workspace (nrf_render_rays_workspace_bytes), with no allocation and no host synchronisation, so a tile
// renderer needs one call per chunk of rays and the call is CUDA-graph capturable.
#include "common.cuh"

namespace nrf {

// The rays of a chunk are adjacent pixels of a frame (GetRays order): the encode kernel walks the same sample of kRayGroup neighbouring rays
// together (nrf_hash_encode_rays_fwd_grouped).
constexpr int kRayGroup = 32;

static inline int64_t align256(int64_t v) { return (v + 255) & ~int64_t(255); }

struct RenderWs {
	int64_t ray_batch, ray_sh, z, z_fine, w_coarse, enc, keep, raw, raw_coarse, perm, rays_d, view_bias, total;
};

static RenderWs render_layout(const nrf_render_config* c, const nrf_hash_grid* g, int64_t R)
{
	RenderWs w;
	const int64_t S = c->n_samples, T = c->n_samples + c->n_importance, D = static_cast<int64_t>(g->n_levels) * g->n_features;
	const int64_t sh = static_cast<int64_t>(c->sh_degree) * c->sh_degree;
	int64_t off = 0;
	w.ray_batch = off; off = align256(off + R * 11 * 4);
	w.ray_sh = off;    off = align256(off + R * sh * 4);
	w.z = off;         off = align256(off + R * S * 4);
	w.z_fine = off;    off = align256(off + R * T * 4);
	w.w_coarse = off;  off = align256(off + R * S * 4);
	w.enc = off;       off = align256(off + R * T * D * 2);
	w.keep = off;      off = align256(off + R * T);
	w.raw = off;       off = align256(off + R * T * 16);
	w.raw_coarse = off; off = align256(off + R * S * 16);
	w.perm = off;      off = align256(off + R * T * 2);
	w.rays_d = off;    off = align256(off + R * 3 * 4);
	w.view_bias = off; off = align256(off + (c->sh_degree != 4 ? R * 64 * 4 : 0));
	w.total = off;
	return w;
}

static int check_render_args(const nrf_render_config* c, const nrf_hash_grid* g)
{
	NRF_REQUIRE(c != nullptr && g != nullptr, "null config / grid");
	NRF_REQUIRE(c->n_samples >= 3 && c->n_importance >= 1, "n_samples must be >= 3 and n_importance >= 1 (SURVEY §9-Q2)");
	NRF_REQUIRE(c->sh_degree >= 1 && c->sh_degree <= 8, "sh_degree out of range");
	return NRF_OK;
}

}  // namespace nrf

using namespace nrf;

extern "C" {

int64_t nrf_render_rays_workspace_bytes(const nrf_render_config* cfg, const nrf_hash_grid* grid, int64_t n_rays)
{
	if (check_render_args(cfg, grid) != NRF_OK || n_rays < 0) return -1;
	return render_layout(cfg, grid, n_rays).total;
}

}

// Where the rays come from: rays_o / rays_d arrays (RenderRays on a ray list); a prepared batch [o d near far viewdirs] (what BatchifyRays hands
// to RenderRays, src/NeRFRenderer.h:483: its near / far / viewdirs are taken as given); or the camera alone (tile: ray r is pixel first_pixel + r
// of an img_w wide image seen through (K, c2w), GetRays, src/RayUtils.h:23-46, inside the prologue kernel).  In the last two cases rays_d lands
// in the workspace for the compositing kernels.
struct RaySrc {
	const float* rays_o; const float* rays_d;                  // arrays
	const float* prepared; int32_t prepared_stride;            // prepared batch
	const float* K_host; const float* c2w_host; int32_t img_w; int64_t first_pixel;   // tile
};

static int render_impl(const nrf_render_config* cfg, const nrf_hash_grid* grid, const void* table_f16, const nrf_mlp_small_shape* shape,
	const void* packed, const RaySrc& src, int64_t n_rays, const float* t_vals, const float* u, void* workspace, int64_t workspace_bytes, float* rgb,
	float* depth, float* disp, float* acc, float* weights, float* z_out, nrf_stream stream)
{
	if (int rc = check_render_args(cfg, grid)) return rc;
	NRF_REQUIRE(n_rays >= 0, "negative n_rays");
	if (n_rays == 0) return NRF_OK;
	const bool tile = src.K_host != nullptr, prepared = src.prepared != nullptr;
	const float* rays_d = src.rays_d;
	NRF_REQUIRE(table_f16 && shape && packed && t_vals && u && workspace, "null pointer");
	NRF_REQUIRE(prepared ? src.prepared_stride >= 11 : (tile ? (src.c2w_host && src.img_w > 0 && src.first_pixel >= 0) : (src.rays_o && src.rays_d)),
		"rays, prepared batch or camera missing");
	NRF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
	const RenderWs w = render_layout(cfg, grid, n_rays);
	NRF_REQUIRE(workspace_bytes >= w.total, "workspace too small (nrf_render_rays_workspace_bytes)");
	const int S = cfg->n_samples, N = cfg->n_importance, T = S + N;
	char* base = static_cast<char*>(workspace);
	float* ray_batch = reinterpret_cast<float*>(base + w.ray_batch);
	float* ray_sh = reinterpret_cast<float*>(base + w.ray_sh);
	float* z = reinterpret_cast<float*>(base + w.z);
	float* z_fine = z_out ? z_out : reinterpret_cast<float*>(base + w.z_fine);
	float* w_coarse = reinterpret_cast<float*>(base + w.w_coarse);
	void* enc = base + w.enc;
	uint8_t* keep = reinterpret_cast<uint8_t*>(base + w.keep);
	float* raw = reinterpret_cast<float*>(base + w.raw);
	float* raw_coarse = reinterpret_cast<float*>(base + w.raw_coarse);
	int16_t* perm = reinterpret_cast<int16_t*>(base + w.perm);
	// One network for both passes (src/NeRFRenderer.h:422,447): the merged fine pass re-uses the coarse pass's raw rows for the coarse
	// samples and gathers / evaluates the importance samples only — the same bits as evaluating all S + N rows (tests/test_gpu_pipeline.py).

	int rc;
	// Render prologue + coarse depths + per-ray SH table: one launch (bit-identical to nrf_rays_prepare + nrf_sh_encode_fwd + nrf_z_sample)
	if (prepared) {
		float* rd = reinterpret_cast<float*>(base + w.rays_d);
		if ((rc = nrf_ray_setup_prepared(src.prepared, src.prepared_stride, n_rays, t_vals, S, cfg->lin_disp, cfg->sh_degree, rd, ray_batch, z, ray_sh, stream)))
			return rc;
		rays_d = rd;
	} else if (tile) {
		float* rd = reinterpret_cast<float*>(base + w.rays_d);
		if ((rc = nrf_ray_setup_tile(src.K_host, src.c2w_host, src.img_w, src.first_pixel, n_rays, cfg->bbox, cfg->near_plane, t_vals, S, cfg->lin_disp,
		                             cfg->sh_degree, nullptr, rd, ray_batch, z, ray_sh, stream))) return rc;
		rays_d = rd;
	} else if ((rc = nrf_ray_setup(src.rays_o, src.rays_d, n_rays, cfg->bbox, cfg->near_plane, t_vals, S, cfg->lin_disp, cfg->sh_degree, ray_batch, z, ray_sh,
	                               nullptr, stream))) return rc;
	// SH degree != 4 (shape->input_ch_views != 16): the view channels enter the network as a per-ray bias, computed once for both passes
	NRF_REQUIRE(shape->input_ch_views == cfg->sh_degree * cfg->sh_degree, "shape->input_ch_views must be sh_degree^2");
	nrf_mlp_input kind = NRF_MLP_IN_ENC16_RAYDIRS;
	const float* views = ray_sh;
	if (shape->input_ch_views != 16) {
		float* vb = reinterpret_cast<float*>(base + w.view_bias);
		if ((rc = nrf_mlp_small_view_bias_fwd(shape, packed, ray_sh, n_rays, vb, nullptr, stream))) return rc;
		kind = NRF_MLP_IN_ENC16_RAYBIAS;
		views = vb;
	}
	// coarse pass
	if ((rc = nrf_hash_encode_rays_fwd_grouped(grid, table_f16, ray_batch, 11, z, n_rays, S, 1, keep, enc, NRF_ENC_F16, nullptr, nullptr, nullptr, 0, kRayGroup, stream)))
		return rc;
	if ((rc = nrf_mlp_small_fwd(shape, packed, kind, enc, views, S, keep, n_rays * S, raw_coarse, stream))) return rc;
	if ((rc = nrf_composite_fwd(raw_coarse, 4, z, rays_d, nullptr, 0.f, cfg->white_bkgr, n_rays, S, nullptr, nullptr, nullptr, nullptr, w_coarse,
	                            stream))) return rc;
	// importance sampling + merge, fine pass
	if ((rc = nrf_sample_pdf_merge_rows(z, w_coarse, u, 0, n_rays, S, N, nullptr, z_fine, perm, raw_coarse, raw, stream))) return rc;
	if ((rc = nrf_hash_encode_rays_fwd_grouped(grid, table_f16, ray_batch, 11, z_fine, n_rays, T, 1, keep, enc, NRF_ENC_F16, perm, nullptr, nullptr, S, kRayGroup,
	                                           stream))) return rc;
	if ((rc = nrf_mlp_small_fwd_importance(shape, packed, kind, enc, views, keep, perm, n_rays, N, T, raw, stream))) return rc;
	if ((rc = nrf_composite_fwd(raw, 4, z_fine, rays_d, nullptr, 0.f, cfg->white_bkgr, n_rays, T, rgb, depth, disp, acc, weights, stream))) return rc;
	return NRF_OK;
}

extern "C" {

int nrf_render_rays_fwd(const nrf_render_config* cfg, const nrf_hash_grid* grid, const void* table_f16, const nrf_mlp_small_shape* shape,
	const void* packed, const float* rays_o, const float* rays_d, int64_t n_rays, const float* t_vals, const float* u, void* workspace,
	int64_t workspace_bytes, float* rgb, float* depth, float* disp, float* acc, float* weights, float* z_out, nrf_stream stream)
{
	NRF_REQUIRE(n_rays <= 0 || (rays_o && rays_d), "null rays");
	const RaySrc src{rays_o, rays_d, nullptr, 0, nullptr, nullptr, 0, 0};
	return render_impl(cfg, grid, table_f16, shape, packed, src, n_rays, t_vals, u, workspace, workspace_bytes, rgb, depth, disp, acc, weights, z_out, stream);
}

int nrf_render_raybatch_fwd(const nrf_render_config* cfg, const nrf_hash_grid* grid, const void* table_f16, const nrf_mlp_small_shape* shape,
	const void* packed, const float* ray_batch, int32_t ray_stride, int64_t n_rays, const float* t_vals, const float* u, void* workspace,
	int64_t workspace_bytes, float* rgb, float* depth, float* disp, float* acc, float* weights, float* z_out, nrf_stream stream)
{
	NRF_REQUIRE(n_rays <= 0 || ray_batch, "null ray batch");
	const RaySrc src{nullptr, nullptr, ray_batch, ray_stride, nullptr, nullptr, 0, 0};
	return render_impl(cfg, grid, table_f16, shape, packed, src, n_rays, t_vals, u, workspace, workspace_bytes, rgb, depth, disp, acc, weights, z_out, stream);
}

int nrf_render_tile_fwd(const nrf_render_config* cfg, const nrf_hash_grid* grid, const void* table_f16, const nrf_mlp_small_shape* shape,
	const void* packed, const float* K_host, const float* c2w_host, int32_t img_w, int64_t first_pixel, int64_t n_rays, const float* t_vals,
	const float* u, void* workspace, int64_t workspace_bytes, float* rgb, float* depth, float* disp, float* acc, float* weights, float* z_out,
	nrf_stream stream)
{
	NRF_REQUIRE(K_host && c2w_host, "null camera");
	const RaySrc src{nullptr, nullptr, nullptr, 0, K_host, c2w_host, img_w, first_pixel};
	return render_impl(cfg, grid, table_f16, shape, packed, src, n_rays, t_vals, u, workspace, workspace_bytes, rgb, depth, disp, acc, weights, z_out, stream);
}

}
