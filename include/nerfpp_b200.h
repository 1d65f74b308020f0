/*
 * nerfpp_b200 — C ABI of the B200-native NeRFpp ray-batch hot path (libnerfpp_b200.so).
 *
 * The reference (DeliriumV01D/NeRFpp) has no FFI: its boundary is C++ template duck-typing
 * (src/NeRFRenderer.h:88-159, src/NeRFExecutor.h:299-301).  The C++ drop-in modules in
 * nerfpp_b200/csrc/host/ keep torch::Tensor at that boundary and call ONLY the functions declared here.
 * Each entry cites the reference code it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller owns every buffer;
 *   - tensors are dense row-major fp32 unless stated; `stream` is a cudaStream_t (NULL = legacy default);
 *   - functions only enqueue work on `stream` (no host sync) and return 0 (NRF_OK) or a negative nrf_status;
 *     nrf_last_error() gives the text for the calling thread;  nothing throws across this ABI;
 *   - no hidden global state besides one-time cudaFuncSetAttribute calls: safe across streams / devices.
 *   - there is NO CPU fallback: without a CUDA device every compute entry returns NRF_ERR_CUDA.
 */
#ifndef NERFPP_B200_H
#define NERFPP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NRF_ABI_VERSION 1

typedef void* nrf_stream; /* cudaStream_t */

typedef enum nrf_status {
	NRF_OK = 0,
	NRF_ERR_INVALID = -1,     /* bad argument (null pointer, unsupported shape) */
	NRF_ERR_CUDA = -2,        /* CUDA runtime / launch error; text in nrf_last_error() */
	NRF_ERR_UNSUPPORTED = -3  /* configuration outside what the sm_100a kernels were built for */
} nrf_status;

int nrf_abi_version(void);
const char* nrf_last_error(void);
/* number of kernel launches issued through this library by the calling process (bench.py "gpu_launches") */
int64_t nrf_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * Multiresolution hash grid — replaces CuHashEmbedderFunction::forward/backward and their kernels
 * (src/CuHashEmbedder.cu:9-102, 106-216, 221-325) and the clamp/keep-mask prologue of
 * CuHashEmbedderImpl::forward (src/CuHashEmbedder.cpp:85-103).
 *
 * The descriptor mirrors the module's public members (src/CuHashEmbedder.h:12-27).  primes / biases /
 * feat_local_idx / feat_local_size are the module's registered buffers, passed as they are (they are saved in
 * checkpoints and pin the hash function, SURVEY §9-Q6).  NOTE feat_local_idx is an offset in SCALARS, not rows
 * (src/CuHashEmbedder.cu:55,150): with F=2 consecutive levels overlap by half — reproduced bit-exactly.
 * ---------------------------------------------------------------------------------------------------------- */
#define NRF_MAX_LEVELS 32

typedef struct nrf_hash_grid {
	int32_t n_levels;           /* NLevels                 (<= NRF_MAX_LEVELS) */
	int32_t n_features;         /* NFeaturesPerLevel       (2, 4 or 8)         */
	int32_t n_volumes;          /* NVolumes                (1)                 */
	int32_t base_resolution;    /* BaseResolution                              */
	int32_t finest_resolution;  /* FinestResolution                            */
	float box_min[3];           /* BoundingBox[0:3]                            */
	float box_max[3];           /* BoundingBox[3:6]                            */
	const int32_t* primes;          /* [n_levels, n_volumes, 3] int32          */
	const float* biases;            /* [n_levels * n_volumes, 3]               */
	const int32_t* feat_local_idx;  /* [n_levels] scalar offsets               */
	const int32_t* feat_local_size; /* [n_levels] entries per level            */
	const float* level_scale;       /* [n_levels] from nrf_hash_level_scales   */
	int64_t table_scalars;          /* numel(Embeddings), for bounds checking  */
} nrf_hash_grid;

/* Per-level scale exp2f((log2f(finest)-log2f(base))*l/(L-1)+log2f(base)), evaluated ON THE DEVICE with the
 * reference's exact expression (src/CuHashEmbedder.cu:40) so floorf() lands on the same cell. */
int nrf_hash_level_scales(int32_t base_resolution, int32_t finest_resolution, int32_t n_levels,
                          float* level_scale, nrf_stream stream);

/* Inspection entry for parity tests: for every (point, level, corner) the SCALAR address into the table (feat_local_idx[level] +
 * hashed position * n_features, src/CuHashEmbedder.cu:55,70-77,150) and the trilinear weight (:83-90), computed by the same device
 * code the encode kernels use; corner order 000,001,...,111 (z fastest).  addr int64 [N, L, 8], weights fp32 [N, L, 8]. */
int nrf_hash_cells(const nrf_hash_grid* grid, const float* points, int64_t n_points, int clamp_points, int64_t* addr,
                   float* weights, nrf_stream stream);

/* fp32 master table -> fp16 shadow, round-to-nearest-even (src/CuHashEmbedder.cu:257). */
int nrf_table_to_half(const float* table_f32, void* table_f16, int64_t n_scalars, nrf_stream stream);

typedef enum nrf_enc_layout {
	NRF_ENC_F32 = 0, /* [N, L*F] fp32 holding fp16-rounded values — what the reference returns (.cu:274) */
	NRF_ENC_F16 = 1  /* [N, L*F] fp16 — same values, fed straight to nrf_mlp_small_* */
} nrf_enc_layout;

/* points [N,3].  clamp_points!=0: clamp into the box and write keep[N] (1 = inside, src/CuHashEmbedder.cpp:92-101;
 * keep may be NULL).  clamp_points==0: points are taken as already clamped. */
int nrf_hash_encode_fwd(const nrf_hash_grid* grid, const void* table_f16, const float* points, int64_t n_points,
                        int clamp_points, uint8_t* keep, void* enc_out, nrf_enc_layout layout, nrf_stream stream);

typedef enum nrf_grad_layout {
	NRF_GRAD_F32 = 0,  /* [N, L*F] fp32 */
	NRF_GRAD_BF16 = 1  /* [N, L*F] bf16 (produced by nrf_mlp_small_bwd) */
} nrf_grad_layout;

/* grad_table[table_scalars] fp32 is ACCUMULATED into (caller zeroes it, or lets nrf_adam_step do so).
 * fp32 accumulation replaces the reference's x128-scaled fp16 atomics (src/CuHashEmbedder.cu:197-198,303,323). */
int nrf_hash_encode_bwd(const nrf_hash_grid* grid, const float* points, int64_t n_points, int clamp_points,
                        const void* grad_enc, nrf_grad_layout layout, float* grad_table, nrf_stream stream);

/* Fused point generation (src/NeRFRenderer.h:419,432 + the two entries above): sample i of ray r is the point
 * o_r + d_r * z[r,i], evaluated inside the kernel with ATen's un-fused rounding (mul, then add) from ray_batch [R, ray_stride]
 * (o at columns 0..2, d at 3..5) and z [R,S]; the [R,S,3] point array is never materialised.  n_rays * n_samples < 2^31.
 *
 * Row reuse (forward only; reuse_perm NULL to disable): reuse_perm [R, S] int16 is nrf_sample_pdf_merge_perm's output for this
 * merged z (S = n_importance + reuse_samples).  The reuse_samples coarse samples whose z it reports as bit-identical are not
 * gathered again: their rows (and keep flags) are copied from the coarse call's output reuse_enc [R, reuse_samples, L*F] (same
 * layout) / reuse_keep [R, reuse_samples] — same point, same table, same bits; all other samples are encoded as usual.
 * reuse_enc NULL: those rows of enc_out (and their keep flags) are left as they are (inference through nrf_mlp_small_fwd_importance,
 * which never reads them). */
int nrf_hash_encode_rays_fwd(const nrf_hash_grid* grid, const void* table_f16, const float* ray_batch, int32_t ray_stride,
                             const float* z, int64_t n_rays, int32_t n_samples, int clamp_points, uint8_t* keep, void* enc_out,
                             nrf_enc_layout layout, const int16_t* reuse_perm, const void* reuse_enc, const uint8_t* reuse_keep,
                             int32_t reuse_samples, nrf_stream stream);
/* Same call, same results; ray_group > 1 only changes the order in which the kernel walks the points: neighbouring lanes take the
 * SAME sample of ray_group neighbouring rays instead of consecutive samples of one ray.  For the rays of a rendered frame
 * (GetRays order: adjacent pixels, src/RayUtils.h:23-46) those points lie a fraction of a fine cell apart and share most corner
 * fetches; for a training batch of random pixels (src/NeRFDataset.cpp:109-144) there is nothing to share: use 1. */
int nrf_hash_encode_rays_fwd_grouped(const nrf_hash_grid* grid, const void* table_f16, const float* ray_batch, int32_t ray_stride,
                                     const float* z, int64_t n_rays, int32_t n_samples, int clamp_points, uint8_t* keep,
                                     void* enc_out, nrf_enc_layout layout, const int16_t* reuse_perm, const void* reuse_enc,
                                     const uint8_t* reuse_keep, int32_t reuse_samples, int32_t ray_group, nrf_stream stream);
int nrf_hash_encode_rays_bwd(const nrf_hash_grid* grid, const float* ray_batch, int32_t ray_stride, const float* z,
                             int64_t n_rays, int32_t n_samples, int clamp_points, const void* grad_enc, nrf_grad_layout layout,
                             float* grad_table, nrf_stream stream);

/* The ray entries above with the per-sample perturbations of the reference's shipped training configuration (src/main.cpp:187
 * thin_ray = false; src/NeRFExecutor.h:411-412 RawNoiseStd / StochasticPreconditioningAlpha) applied inside the kernels, in the order of
 * src/NeRFRenderer.h:419-445:
 *     p = o + d z                                                     (:419 / :432)
 *     sp_noise != NULL:   p = ReflectBoundary(p + sp_noise * alpha)   (:435-443, :285-304; the caller passes it for the fine pass only)
 *     cone_angle != NULL: p += (t r cos(theta) + b r sin(theta)) * cone_angle * z, then clamped into the grid's box if clamp_to_box
 *                                                                     (TangentScatter, :307-362)
 * then the encode's own clamp / keep mask as above.  This replaces nrf_sample_points -> nrf_precondition_points -> nrf_tangent_scatter ->
 * nrf_hash_encode_fwd / _bwd on the [R,S,3] array, with the same arithmetic (bit-identical points); no point array exists in either
 * direction: the backward re-derives the forward's points from the same variates.  The variates are the caller's torch draws, so the
 * Philox stream stays the reference's.  No row reuse (a jittered sample is re-jittered with fresh draws in the fine pass). */
typedef struct nrf_point_jitter {
	const float* cone_angle;   /* NULL = thin rays; one scalar (cone_stride 0) or one per ray at cone_angle[ray * cone_stride]         */
	int32_t cone_stride;
	const float* rand_r;       /* [R,S] uniforms: the two torch::rand draws of src/NeRFRenderer.h:342-343 (needed with a cone)          */
	const float* rand_theta;
	int32_t clamp_to_box;      /* TangentScatter's clamp into the grid's box (bounding box given, :356-360)                            */
	const float* sp_noise;     /* [R,S,3] standard normal (randn_like(pts), :437); NULL = no stochastic preconditioning                 */
	const float* sp_alpha;     /* DEVICE scalar: the step's StochasticPreconditioningAlpha (needed with sp_noise)                      */
} nrf_point_jitter;

int nrf_hash_encode_rays_jitter_fwd(const nrf_hash_grid* grid, const void* table_f16, const float* ray_batch, int32_t ray_stride,
                                    const float* z, int64_t n_rays, int32_t n_samples, int clamp_points, uint8_t* keep, void* enc_out,
                                    nrf_enc_layout layout, const nrf_point_jitter* jitter, nrf_stream stream);
int nrf_hash_encode_rays_jitter_bwd(const nrf_hash_grid* grid, const float* ray_batch, int32_t ray_stride, const float* z,
                                    int64_t n_rays, int32_t n_samples, int clamp_points, const void* grad_enc, nrf_grad_layout layout,
                                    float* grad_table, const nrf_point_jitter* jitter, nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * Direction / position encoders
 * ---------------------------------------------------------------------------------------------------------- */
/* CuSHKernel (src/CuSHEncoder.cu:4-107): dirs -> [N, degree^2], degree 1..8.  Direction i is read at
 * dirs + i*dir_stride (3 for the reference's contiguous [N,3]; 11 reads the viewdirs straight out of a ray_batch). */
int nrf_sh_encode_fwd(const float* dirs, int32_t dir_stride, int64_t n, int32_t degree, float* out, nrf_stream stream);

/* EmbedderImpl::forward (src/NeRF.cpp:22-39): x [N,D] -> [N, D*(include_input + 2*num_freqs)],
 * channel order x, sin(f0 x), cos(f0 x), sin(f1 x) ...; freq_bands_host[num_freqs] as built at src/NeRF.cpp:11-19. */
int nrf_posenc_fwd(const float* x, int64_t n, int32_t input_dims, int32_t num_freqs, const float* freq_bands_host,
                   int32_t include_input, float* out, nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * NeRFSmall (HashNeRF MLP) — NeRFSmallImpl::forward (src/NeRF.cpp:363-412) and its autograd backward.
 * Built for the BASELINE shape: sigma net in->64->(1+15), colour net (views+15)->64->64->3, bias-free, ReLU
 * between layers only, output [rgb(3), sigma].  Other shapes return NRF_ERR_UNSUPPORTED.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct nrf_mlp_small_shape {
	int32_t input_ch;          /* 32  (hash L*F)             */
	int32_t input_ch_views;    /* 16  (SH degree 4); 1..64 via NRF_MLP_IN_ENC16_RAYBIAS */
	int32_t hidden_dim;        /* 64                          */
	int32_t geo_feat_dim;      /* 15                          */
	int32_t hidden_dim_color;  /* 64                          */
	int32_t num_layers;        /* 2                           */
	int32_t num_layers_color;  /* 3                           */
} nrf_mlp_small_shape;

/* bytes of the packed (tensor-core fragment ordered, bf16/fp16) weight blob */
int64_t nrf_mlp_small_packed_bytes(const nrf_mlp_small_shape* shape);
/* number of fp32 scalars in the flat parameter / gradient vector, order sigma_net_0, sigma_net_1,
 * color_net_0, color_net_1, color_net_2, each [out, in] row-major (= torch Linear.weight, src/NeRF.cpp:338-342) */
int64_t nrf_mlp_small_param_count(const nrf_mlp_small_shape* shape);
int nrf_mlp_small_pack(const nrf_mlp_small_shape* shape, const float* params_flat, void* packed, nrf_stream stream);

typedef enum nrf_mlp_input {
	NRF_MLP_IN_ENC16_RAYDIRS = 0, /* enc: fp16 [N,32]; views: per-ray SH table fp32 [R,16]; row n uses ray n / samples_per_ray */
	NRF_MLP_IN_F32_CAT = 1,       /* enc: fp32 [N, input_ch + input_ch_views] = cat(embedded, embedded_dirs) (src/NeRFRenderer.h:182) */
	NRF_MLP_IN_ENC16_RAYBIAS = 2  /* enc: fp16 [N,32]; the view channels enter as a per-RAY bias of the colour net's first layer: the "ray_sh" argument is
	                                 bias [R,64] fp32 = nrf_mlp_small_view_bias_fwd's output; row n uses ray n / samples_per_ray.  Any input_ch_views in
	                                 1..64 (SH degree 1..8; 64 = the shipped degree 8, src/main.cpp:176); the other two kinds are built for 16 */
} nrf_mlp_input;

/* keep (nullable): sigma := 0 where keep==0 (src/NeRFRenderer.h:187-188).  raw_out [N,4] = [r,g,b,sigma]. */
int nrf_mlp_small_fwd(const nrf_mlp_small_shape* shape, const void* packed, nrf_mlp_input in_kind, const void* enc,
                      const float* ray_sh, int32_t samples_per_ray, const uint8_t* keep, int64_t n,
                      float* raw_out, nrf_stream stream);

/* The fine pass of RenderRays when coarse and fine share one network (src/NeRFRenderer.h:422,447; src/NeRFExecutor.h:882-890):
 * only the n_importance NEW samples of each ray are evaluated.  Work row (ray, j < n_importance) reads its fp16 encoding at row
 * perm[ray, j] of enc_merged [R, n_merged, 32] (keep_merged [R, n_merged], nullable, likewise; views: ray_sh [R,16]) and writes
 * raw_merged [R, n_merged, 4] at the same row.  perm [R, n_merged] int16 = nrf_sample_pdf_merge_perm's output; the coarse
 * samples' rows of raw_merged are the coarse pass's own rows, moved there by nrf_sample_pdf_merge_rows — the same bits a full
 * nrf_mlp_small_fwd over the merged rows produces (rows are independent), at n_importance / n_merged of its work. */
int nrf_mlp_small_fwd_importance(const nrf_mlp_small_shape* shape, const void* packed, nrf_mlp_input in_kind, const void* enc_merged,
                                 const float* ray_sh, const uint8_t* keep_merged, const int16_t* perm, int64_t n_rays,
                                 int32_t n_importance, int32_t n_merged, float* raw_merged, nrf_stream stream);

/* The view term of the colour net's first layer (src/NeRF.cpp:383-392: h = cat([input_views, geo_feat]) -> Linear) depends on the ray only:
 * bias_out[r, n] = sum_k ray_sh[r, k] W[n, k] over the input_ch_views columns of color_net_0's weight (the packed blob carries an fp32
 * copy of that block), fp32.  Computed once per ray batch, shared by the coarse and the fine pass, and handed to the fused
 * kernels as NRF_MLP_IN_ENC16_RAYBIAS.  grad_bias_zero (nullable) [R,64]: zeroed by the same launch (the accumulator of _bwd_raybias). */
int nrf_mlp_small_view_bias_fwd(const nrf_mlp_small_shape* shape, const void* packed, const float* ray_sh, int64_t n_rays,
                                float* bias_out, float* grad_bias_zero, nrf_stream stream);
/* ... and its weight gradient: grad_params_flat[color_net_0 view columns] += grad_bias^T ray_sh, with grad_bias [R,64] accumulated by
 * nrf_mlp_small_bwd_raybias (the per-ray sum of the gradient at that layer's pre-activation). */
int nrf_mlp_small_view_bias_bwd(const nrf_mlp_small_shape* shape, const float* ray_sh, const float* grad_bias, int64_t n_rays,
                                float* grad_params_flat, nrf_stream stream);

/* grad_raw [N,4].  grad_in: bf16 [N,32] (NRF_MLP_IN_ENC16_RAYDIRS) or fp32 [N,48] (NRF_MLP_IN_F32_CAT), may be NULL.
 * grad_params_flat[param_count] fp32 is ACCUMULATED into.  Activations are recomputed, nothing was saved. */
int nrf_mlp_small_bwd(const nrf_mlp_small_shape* shape, const void* packed, nrf_mlp_input in_kind, const void* enc,
                      const float* ray_sh, int32_t samples_per_ray, const uint8_t* keep, int64_t n,
                      const float* grad_raw, void* grad_in, float* grad_params_flat, nrf_stream stream);
/* Same for every in_kind; NRF_MLP_IN_ENC16_RAYBIAS additionally needs grad_bias [R,64] fp32 (ACCUMULATED into: per-ray sums of the gradient
 * at the colour net's first pre-activation; samples_per_ray % 16 == 0) — the view columns of color_net_0's gradient then come from
 * nrf_mlp_small_view_bias_bwd.  grad_bias is ignored (may be NULL) for the other kinds. */
int nrf_mlp_small_bwd_raybias(const nrf_mlp_small_shape* shape, const void* packed, nrf_mlp_input in_kind, const void* enc,
                              const float* ray_sh, int32_t samples_per_ray, const uint8_t* keep, int64_t n,
                              const float* grad_raw, void* grad_in, float* grad_params_flat, float* grad_bias, nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * Classic NeRF MLP, forward (inference) — NeRFImpl::forward (src/NeRF.cpp:92-126) fused on tcgen05 tensor cores: 8 x 256 ReLU
 * layers with the skip concat [x | h] after layer 4 (:103-104), alpha head (:110), feature layer (:111), view branch
 * [feature | dirs] -> 128 -> ReLU -> rgb (:112-119), biases included, out = [rgb(3), alpha] (:120).  Built for the BASELINE
 * shape (NeRFExecutor.h:478: D=8, W=256, input_ch=63, input_ch_views=27, skips={4}, use_viewdirs); other shapes return
 * NRF_ERR_UNSUPPORTED.  x [N, 90] fp32 = cat(embedded points, embedded dirs) (src/NeRFRenderer.h:182), out [N,4] fp32.
 *
 * Training (the autograd backward of the same forward, src/NeRFExecutor.h:883-890 -> loss.backward()):
 *   nrf_mlp_nerf_pack_train   bf16 copy of the weights in the same blob layout (bf16 keeps fp32's exponent range: with the
 *                             reference's Xavier(0.1) initialisation, Trainable.h:43, fp16 activations of the deep layers are 0)
 *   nrf_mlp_nerf_fwd_train    the forward on that blob; additionally stores every layer's input, bf16, into `saved`
 *                             (nrf_mlp_nerf_saved_bytes(n) bytes, 128-byte aligned)
 *   nrf_mlp_nerf_bwd          grad_out [N,4] fp32 (d loss / d [rgb, alpha]) -> gradients of the 12 weight matrices and biases,
 *                             ADDED (+=, fp32 atomics) to the caller's tensors in torch Linear layout; `workspace` needs
 *                             nrf_mlp_nerf_bwd_workspace_bytes(n) bytes.  No gradient with respect to x is produced: the
 *                             positional embedder feeding x has no parameters (src/NeRF.cpp:4-39).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct nrf_mlp_nerf_shape {
	int32_t depth;           /* 8   */
	int32_t width;           /* 256 */
	int32_t input_ch;        /* 63  */
	int32_t input_ch_views;  /* 27  */
	int32_t skip_layer;      /* 4   */
	int32_t use_viewdirs;    /* 1   */
} nrf_mlp_nerf_shape;

typedef struct nrf_mlp_nerf_weights {   /* device pointers, torch Linear layout [out, in] row-major fp32 (src/NeRF.cpp:52-75) */
	const float* pts_w[8];
	const float* pts_b[8];
	const float* feature_w; const float* feature_b;
	const float* alpha_w;   const float* alpha_b;
	const float* views_w;   const float* views_b;
	const float* rgb_w;     const float* rgb_b;
} nrf_mlp_nerf_weights;

int64_t nrf_mlp_nerf_packed_bytes(const nrf_mlp_nerf_shape* shape);
int nrf_mlp_nerf_pack(const nrf_mlp_nerf_shape* shape, const nrf_mlp_nerf_weights* weights, void* packed, nrf_stream stream);
int nrf_mlp_nerf_fwd(const nrf_mlp_nerf_shape* shape, const void* packed, const float* x, int64_t n, float* out, nrf_stream stream);

typedef struct nrf_mlp_nerf_grads {     /* device pointers, same shapes as nrf_mlp_nerf_weights; accumulated into */
	float* pts_w[8];
	float* pts_b[8];
	float* feature_w; float* feature_b;
	float* alpha_w;   float* alpha_b;
	float* views_w;   float* views_b;
	float* rgb_w;     float* rgb_b;
} nrf_mlp_nerf_grads;

int nrf_mlp_nerf_pack_train(const nrf_mlp_nerf_shape* shape, const nrf_mlp_nerf_weights* weights, void* packed_train, nrf_stream stream);
int64_t nrf_mlp_nerf_saved_bytes(const nrf_mlp_nerf_shape* shape, int64_t n);
int64_t nrf_mlp_nerf_bwd_workspace_bytes(const nrf_mlp_nerf_shape* shape, int64_t n);
int nrf_mlp_nerf_fwd_train(const nrf_mlp_nerf_shape* shape, const void* packed_train, const float* x, int64_t n, float* out, void* saved,
                           nrf_stream stream);
int nrf_mlp_nerf_bwd(const nrf_mlp_nerf_shape* shape, const void* packed_train, const void* saved, const float* grad_out, int64_t n,
                     void* workspace, const nrf_mlp_nerf_grads* grads, nrf_stream stream);

/* The same two forwards fed with what NeRFRenderer::RunNetwork (src/NeRFRenderer.h:164-194) starts from: sample positions
 * points [N,3] and ray directions dirs [R,3] (row n belongs to ray n / samples_per_ray; the reference expands the directions per
 * sample, :179-181).  The positional embeddings of both (EmbedderImpl::forward, src/NeRF.cpp:22-39, frequency bands passed from the
 * host: 10 for points, 4 for directions — the BASELINE multires) are evaluated inside the kernel's input stage with the arithmetic of
 * nrf_posenc_fwd, so the result is bit-identical to nrf_posenc_fwd x 2 + concatenation (:182) + nrf_mlp_nerf_fwd[_train] without the
 * [N,63], [N,27] and [N,90] arrays.  nrf_mlp_nerf_bwd is unchanged (it never reads x). */
int nrf_mlp_nerf_fwd_points(const nrf_mlp_nerf_shape* shape, const void* packed, const float* points, const float* dirs, int32_t samples_per_ray,
                            const float* freqs_pts_host, int32_t n_freqs_pts, const float* freqs_views_host, int32_t n_freqs_views, int64_t n,
                            float* out, nrf_stream stream);
int nrf_mlp_nerf_fwd_train_points(const nrf_mlp_nerf_shape* shape, const void* packed_train, const float* points, const float* dirs,
                                  int32_t samples_per_ray, const float* freqs_pts_host, int32_t n_freqs_pts, const float* freqs_views_host,
                                  int32_t n_freqs_views, int64_t n, float* out, void* saved, nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * Volume rendering — NeRFRenderer::RawToOutputs (src/NeRFRenderer.h:199-282) with TruncExp
 * (src/CustomOps.cpp:5-16) folded in, and its backward.
 * raw [R,S,raw_stride] (channels 0..2 rgb logits, 3 density), z [R,S], rays_d [R,3],
 * noise (nullable) [R,S] standard normal scaled by raw_noise_std (src/NeRFRenderer.h:253-254).
 * ---------------------------------------------------------------------------------------------------------- */
int nrf_composite_fwd(const float* raw, int32_t raw_stride, const float* z, const float* rays_d, const float* noise,
                      float raw_noise_std, int32_t white_bkgr, int64_t n_rays, int32_t n_samples,
                      float* rgb /*[R,3]*/, float* depth /*[R]*/, float* disp /*[R]*/, float* acc /*[R]*/,
                      float* weights /*[R,S] nullable*/, nrf_stream stream);

/* g_* are the upstream gradients of the five outputs (each nullable = zero).  d_raw [R,S,4].  n_samples <= 2048 (register-resident
 * kernels up to 256 samples per ray, a two-pass kernel beyond). */
int nrf_composite_bwd(const float* raw, int32_t raw_stride, const float* z, const float* rays_d, const float* noise,
                      float raw_noise_std, int32_t white_bkgr, int64_t n_rays, int32_t n_samples,
                      const float* g_rgb, const float* g_depth, const float* g_disp, const float* g_acc,
                      const float* g_weights, float* d_raw, nrf_stream stream);

/* The training tail of the colour pass in ONE launch: RawToOutputs forward of every ray, huber_loss(RGBMap, target, delta) with mean reduction
 * over the R*3 values (src/NeRFExecutor.h:883-886) and the backward of both — equal to nrf_composite_fwd -> nrf_huber_fwd_bwd ->
 * nrf_composite_bwd(g_rgb).  loss_out[0] += loss (caller zeroes), rgb_out [R,3] (nullable) the RGBMap, d_raw [R,S,4] = d (loss * grad_scale) / d raw. */
int nrf_composite_huber_bwd(const float* raw, int32_t raw_stride, const float* z, const float* rays_d, const float* noise,
                            float raw_noise_std, int32_t white_bkgr, int64_t n_rays, int32_t n_samples, const float* target, float delta,
                            float grad_scale, float* loss_out, float* rgb_out, float* d_raw, nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * Hierarchical resampling — SamplePDF (src/Sampler.h:6-43).
 * bins [R,B], weights [R,B-1], u: [n_samples] shared (det: linspace(0,1,n), src/Sampler.h:20) when u_per_ray==0,
 * else [R,n_samples].  samples_out [R,n_samples].
 * ---------------------------------------------------------------------------------------------------------- */
int nrf_sample_pdf(const float* bins, const float* weights, int32_t n_bins, const float* u, int32_t u_per_ray,
                   int64_t n_rays, int32_t n_samples, float* samples_out, nrf_stream stream);

/* The fused call site in RenderRays (src/NeRFRenderer.h:427-431): z_mid, SamplePDF(z_mid, w[:,1:-1]), then
 * sort(cat(z, z_samples)).  Both lists are already sorted, so the sort is a rank merge.
 * z_coarse [R,S], weights [R,S] -> z_merged [R,S+n_importance]; z_samples (nullable) [R,n_importance]. */
int nrf_sample_pdf_merge(const float* z_coarse, const float* weights, const float* u, int32_t u_per_ray,
                         int64_t n_rays, int32_t n_samples, int32_t n_importance, float* z_samples,
                         float* z_merged, nrf_stream stream);

/* Same, and perm_out [R, n_importance + S] int16 (nullable): entry j < n_importance is the merged position of the j-th
 * importance sample (in sorted order); entry n_importance + k is the merged position p of coarse sample k, with z_merged[r,p]
 * bit-identical to z_coarse[r,k] (on rays whose fp32 z is not monotone — ones that miss the box — the sample goes to the sorted
 * rank of its value).  u_per_ray != 0 re-sorts everything and reports -(p+1) for every coarse sample: nothing is reusable. */
int nrf_sample_pdf_merge_perm(const float* z_coarse, const float* weights, const float* u, int32_t u_per_ray,
                              int64_t n_rays, int32_t n_samples, int32_t n_importance, float* z_samples,
                              float* z_merged, int16_t* perm_out, nrf_stream stream);

/* Same, and (u shared by the rays only) the coarse pass's raw rows travel with their samples: rows_coarse [R,S,4] f32 ->
 * rows_merged [R,S+n_importance,4] at the merged positions of the coarse samples.  The reference uses ONE network for the coarse
 * and the fine pass (src/NeRFRenderer.h:422,447; src/NeRFExecutor.h:882-890), so these are the fine pass's raw rows for those
 * samples bit for bit; nrf_mlp_small_fwd_importance fills in the importance samples.  Both pointers NULL: as _perm. */
int nrf_sample_pdf_merge_rows(const float* z_coarse, const float* weights, const float* u, int32_t u_per_ray,
                              int64_t n_rays, int32_t n_samples, int32_t n_importance, float* z_samples,
                              float* z_merged, int16_t* perm_out, const float* rows_coarse, float* rows_merged,
                              nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * Rays — RayUtils / Render prologue
 * ---------------------------------------------------------------------------------------------------------- */
/* GetRays (src/RayUtils.h:5-46) for image rows [row_begin,row_end): K_host[9] row-major 3x3, c2w_host[12] = c2w[:3,:4].
 * rays_o, rays_d [(row_end-row_begin)*w, 3]. */
int nrf_get_rays(int32_t h, int32_t w, const float* K_host, const float* c2w_host, int32_t row_begin, int32_t row_end,
                 float* rays_o, float* rays_d, nrf_stream stream);

/* Render prologue (src/NeRFRenderer.h:549-583): viewdirs = d/|d|, near/far = IntersectWithAABB(o,d,bbox,near_plane)
 * (src/RayUtils.h:87-126), ray_batch [R, 8 or 11] = [o, d, near, far (, viewdirs)]. */
int nrf_rays_prepare(const float* rays_o, const float* rays_d, int64_t n_rays, const float* bbox_host /*[6]*/,
                     float near_plane, int32_t use_viewdirs, float* ray_batch, nrf_stream stream);

/* nrf_rays_prepare (with viewdirs) + nrf_z_sample + nrf_sh_encode_fwd(viewdirs) in ONE launch — the head of every RenderRays call
 * (src/NeRFRenderer.h:549-583, :393-402, CuSHEncoder per ray) — bit-identical to the three separate entries.  ray_batch [R,11],
 * z [R,S], ray_sh [R, sh_degree^2] (nullable), zero_scalar (nullable): one float set to 0 (the training step's loss accumulator). */
int nrf_ray_setup(const float* rays_o, const float* rays_d, int64_t n_rays, const float* bbox_host /*[6]*/, float near_plane,
                  const float* t_vals, int32_t n_samples, int32_t lin_disp, int32_t sh_degree, float* ray_batch, float* z, float* ray_sh,
                  float* zero_scalar, nrf_stream stream);

/* NeRFDataset::GetRayBatch (src/NeRFDataset.cpp:109-144) and the target gather of NeRFDataset::get_batch (:156) on the device: pix_hw int32
 * [R,2] = (row, column) of every sampled pixel (the reference draws them with torch::randint, :154-155) -> rays_o, rays_d [R,3] (the
 * GetRays arithmetic at that pixel, bit for bit) and, when image fp32 [img_h, img_w, img_c] is given, target [R, img_c] = image[row, col].
 * cone_angle_host (nullable): the scalar the reference returns, (1/fx + 1/fy) / 2 (:136-141). */
int nrf_ray_batch(const int32_t* pix_hw, int64_t n_rays, const float* K_host, const float* c2w_host, const float* image, int32_t img_h,
                  int32_t img_w, int32_t img_c, float* rays_o, float* rays_d, float* target, float* cone_angle_host, nrf_stream stream);

/* nrf_ray_batch + nrf_ray_setup in ONE launch: a training step then needs (pixel indices, K, c2w) instead of host-generated rays and
 * targets.  rays_o / rays_d / target are OUTPUTS (the compositing and loss kernels read them). */
int nrf_ray_setup_pixels(const int32_t* pix_hw, int64_t n_rays, const float* K_host, const float* c2w_host, const float* image, int32_t img_h,
                         int32_t img_w, int32_t img_c, const float* bbox_host, float near_plane, const float* t_vals, int32_t n_samples,
                         int32_t lin_disp, int32_t sh_degree, float* rays_o, float* rays_d, float* target, float* ray_batch, float* z,
                         float* ray_sh, float* zero_scalar, nrf_stream stream);

/* The same prologue for a tile of a frame: ray r is pixel first_pixel + r in GetRays order (src/RayUtils.h:23-46) of an img_w wide view.
 * rays_o (nullable) / rays_d [R,3] are outputs. */
int nrf_ray_setup_tile(const float* K_host, const float* c2w_host, int32_t img_w, int64_t first_pixel, int64_t n_rays,
                       const float* bbox_host, float near_plane, const float* t_vals, int32_t n_samples, int32_t lin_disp,
                       int32_t sh_degree, float* rays_o, float* rays_d, float* ray_batch, float* z, float* ray_sh, nrf_stream stream);

/* The same prologue for an already prepared ray batch (rows [o d near far viewdirs], ray_stride >= 11): z from its near / far, the SH table
 * from its viewdirs; rays_d [R,3] and the packed [R,11] ray_batch are outputs. */
int nrf_ray_setup_prepared(const float* ray_batch_in, int32_t ray_stride, int64_t n_rays, const float* t_vals, int32_t n_samples,
                           int32_t lin_disp, int32_t sh_degree, float* rays_d, float* ray_batch, float* z, float* ray_sh, nrf_stream stream);

/* z = near*(1-t)+far*t (or the lin_disp variant), src/NeRFRenderer.h:393-402.  t_vals [S] device. */
int nrf_z_sample(const float* ray_batch, int32_t ray_stride, const float* t_vals, int64_t n_rays, int32_t n_samples,
                 int32_t lin_disp, float* z, nrf_stream stream);

/* pts = o + d*z, src/NeRFRenderer.h:419,432.  pts [R,S,3]. */
int nrf_sample_points(const float* ray_batch, int32_t ray_stride, const float* z, int64_t n_rays, int32_t n_samples,
                      float* pts, nrf_stream stream);

/* Stochastic preconditioning (src/NeRFRenderer.h:435-443) + ReflectBoundary (:285-304), in place: pts [N,3] += noise [N,3] * alpha, folded back
 * into bbox_host[6] by reflection.  noise: the reference's torch::randn_like(pts) draw, supplied by the caller. */
int nrf_precondition_points(float* pts, const float* noise, float alpha, const float* bbox_host, int64_t n_points, nrf_stream stream);

/* TangentScatter (src/NeRFRenderer.h:307-362): pts [R,S,3] += (tangent*r*cos(theta) + bitangent*r*sin(theta)) * cone_angle*z,
 * then clamp into bbox_host[6] (nullable = no clamp).  rand_r / rand_theta [R,S] are the two torch::rand draws of :342-343
 * (drawn by the host so the RNG stream matches the reference's).  cone_angle: one scalar (cone_stride 0) or one per ray
 * at cone_angle[ray*cone_stride].  Directions are read at rays_d + ray*dir_stride. */
int nrf_tangent_scatter(float* pts, const float* z, const float* cone_angle, int32_t cone_stride, const float* rays_d,
                        int32_t dir_stride, const float* rand_r, const float* rand_theta, const float* bbox_host,
                        int64_t n_rays, int32_t n_samples, nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * RenderRays for inference in one call — NeRFRenderer::RenderRays (src/NeRFRenderer.h:366-459) behind the Render prologue
 * (:549-583) for <CuHashEmbedder, CuSHEncoder, NeRFSmall>, parity configuration (ThinRay, Perturb 0, no raw noise): ray prologue,
 * SH per ray, z sampling, [hash encode + fused MLP], RawToOutputs, SamplePDF + merge, second network pass, RawToOutputs.
 * Enqueues this library's kernels on `stream` into a caller-owned workspace; no allocation, no host sync (graph-capturable).
 * t_vals [n_samples] = linspace(0,1) (src/NeRFRenderer.h:393) and u [n_importance] = linspace(0,1) (src/Sampler.h:20) are device
 * arrays.  Outputs: rgb [R,3], depth/disp/acc [R], weights / z_out [R, n_samples+n_importance] (each nullable).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct nrf_render_config {
	int32_t n_samples;      /* NSamples                        */
	int32_t n_importance;   /* NImportance (>= 1, SURVEY Q2)  */
	int32_t white_bkgr;     /* WhiteBkgr                       */
	int32_t lin_disp;       /* LinDisp                         */
	int32_t sh_degree;      /* CuSHEncoder degree (4)          */
	float near_plane;       /* IntersectWithAABB near clamp    */
	float bbox[6];          /* BoundingBox (host)              */
} nrf_render_config;

int64_t nrf_render_rays_workspace_bytes(const nrf_render_config* cfg, const nrf_hash_grid* grid, int64_t n_rays);
int nrf_render_rays_fwd(const nrf_render_config* cfg, const nrf_hash_grid* grid, const void* table_f16,
                        const nrf_mlp_small_shape* shape, const void* packed, const float* rays_o, const float* rays_d,
                        int64_t n_rays, const float* t_vals, const float* u, void* workspace, int64_t workspace_bytes,
                        float* rgb, float* depth, float* disp, float* acc, float* weights, float* z_out, nrf_stream stream);

/* The same for a tile of a frame given only the camera (SURVEY §8f-3: Render(h, w, K, c2w), src/NeRFRenderer.h:540-547 with GetRays,
 * src/RayUtils.h:23-46, fused into the prologue kernel): ray r is pixel first_pixel + r in GetRays order (row-major, img_w wide) of the
 * view (K_host[9] row-major 3x3, c2w_host[12] = c2w[:3,:4]).  No rays_o / rays_d arrays exist; same results as nrf_get_rays +
 * nrf_render_rays_fwd bit for bit.  Workspace: nrf_render_rays_workspace_bytes(cfg, grid, n_rays). */
int nrf_render_tile_fwd(const nrf_render_config* cfg, const nrf_hash_grid* grid, const void* table_f16,
                        const nrf_mlp_small_shape* shape, const void* packed, const float* K_host, const float* c2w_host,
                        int32_t img_w, int64_t first_pixel, int64_t n_rays, const float* t_vals, const float* u, void* workspace,
                        int64_t workspace_bytes, float* rgb, float* depth, float* disp, float* acc, float* weights, float* z_out,
                        nrf_stream stream);

/* The same for a prepared ray batch — rows [o(3) d(3) near far viewdirs(3) ...] of ray_stride >= 11 floats, what BatchifyRays hands to RenderRays
 * (src/NeRFRenderer.h:483, built by Render :549-583): near / far / viewdirs are taken from the batch, cfg->bbox / near_plane are not used.
 * This is the call the drop-in NeRFRenderer::RenderRays makes when no autograd graph is recorded (host/renderer.h). */
int nrf_render_raybatch_fwd(const nrf_render_config* cfg, const nrf_hash_grid* grid, const void* table_f16,
                            const nrf_mlp_small_shape* shape, const void* packed, const float* ray_batch, int32_t ray_stride,
                            int64_t n_rays, const float* t_vals, const float* u, void* workspace, int64_t workspace_bytes,
                            float* rgb, float* depth, float* disp, float* acc, float* weights, float* z_out, nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training glue restated from NeRFExecutor::Train (src/NeRFExecutor.h:883-890, 539, 986)
 * ---------------------------------------------------------------------------------------------------------- */
/* huber_loss(pred, target, delta=1, mean): loss_out[0] += mean loss (caller zeroes), grad[n] = dLoss/dpred * grad_scale */
int nrf_huber_fwd_bwd(const float* pred, const float* target, int64_t n, float delta, float grad_scale,
                      float* loss_out, float* grad, nrf_stream stream);

/* torch::optim::Adam step (no amsgrad, no weight decay): g = grad*grad_scale; m,v updated; bias-corrected update.
 * step is 1-based.  zero_grad!=0 clears grad afterwards.  shadow_f16 (nullable): fp16 copy of the new params
 * (replaces the per-forward full-table cast, src/CuHashEmbedder.cu:257). */
int nrf_adam_step(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                  float beta2, float eps, int32_t step, float grad_scale, int32_t zero_grad, void* shadow_f16,
                  nrf_stream stream);

/* CUDA-graph replay of the optimiser: the step count, Adam bias corrections and the decayed learning rate
 * lr0 * decay_rate^(max(step-2,0) / decay_steps) (src/NeRFExecutor.h:992-996, evaluated in the order of :986-996) live in a
 * 16-byte device record {int32 step; float lr/(1-b1^step); float 1/sqrt(1-b2^step); float lr}, zero-initialised by the caller.
 * nrf_adam_schedule_advance increments it ON THE DEVICE (fp64 arithmetic); nrf_adam_step_scheduled is nrf_adam_step reading it.
 * Both only enqueue work, so one captured graph replays every training step. */
int nrf_adam_schedule_advance(void* sched_state, float lr0, float decay_rate, float decay_steps, float beta1, float beta2,
                              nrf_stream stream);
int nrf_adam_step_scheduled(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const void* sched_state,
                            float beta1, float beta2, float eps, float grad_scale, int32_t zero_grad, void* shadow_f16,
                            nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * Data-parallel optimiser step fused with its collectives over NVLink peer memory (no counterpart in the reference, which
 * is single-GPU): reduce-scatter of the flat gradient + Adam on this rank's 1/world shard + all-gather of the fp16 shadow,
 * ONE kernel per rank.  All pointer arrays hold addresses valid on THIS device for every rank's buffer (peer-mapped, e.g.
 * torch.distributed._symmetric_memory buffer_ptrs); entry [rank] is the local one.
 *   grads[p]       fp32 [n_total]  rank p's local gradient (summed in rank order, cleared locally at the end)
 *   shadow_f16[p]  fp16 [n_total]  rank p's parameter shadow (the owner of a scalar writes its new value to every rank)
 *   flags[p]       nrf_peer_flags_bytes(world) bytes, zero-initialised once (system-scope barrier words and epoch)
 * The first n_sharded scalars (the hash table) are owned in contiguous shards of floor/ceil(n_sharded/4/world) quads; the
 * tail [n_sharded, n_total) (the MLP weights) is updated identically on every rank.  param/exp_avg/exp_avg_sq are local
 * fp32 [n_total]; only the owned shard and the tail are touched (non-owned table entries of `param` go stale by design:
 * the forward reads the shadow).  Every rank must call this once per step; a missing peer releases the others after ~2 s.
 * ---------------------------------------------------------------------------------------------------------- */
#define NRF_MAX_PEERS 8
typedef struct nrf_peer_group {
	int32_t world, rank;
	const float* grads[NRF_MAX_PEERS];
	void* shadow_f16[NRF_MAX_PEERS];
	uint32_t* flags[NRF_MAX_PEERS];
	/* optional NVSwitch multicast mappings of the SAME two buffers (NULL: peer loads / stores on the pointers above): one address that
	 * reads the sum over all ranks (multimem.ld_reduce: the reduction happens in the switch, each element crosses this GPU's link once
	 * instead of world - 1 times) / writes every rank's copy (multimem.st) */
	const float* grads_mc;
	void* shadow_f16_mc;
} nrf_peer_group;

int64_t nrf_peer_flags_bytes(int32_t world);
int nrf_adam_step_sharded(const nrf_peer_group* pg, float* param, float* exp_avg, float* exp_avg_sq, int64_t n_sharded,
                          int64_t n_total, const void* sched_state, float beta1, float beta2, float eps, float grad_scale,
                          nrf_stream stream);

/* ------------------------------------------------------------------------------------------------------------
 * LeRF language head (SURVEY §8f-1, BASELINE C5) — LeRFImpl::forward (src/LeRF.cpp:28-111), the keep mask of
 * LeRFRenderer::RunLENetwork (src/LeRFRenderer.cpp:18-20) and RenderCLIPEmbedding (src/LeRFRenderer.h:45-54), fused on tcgen05
 * tensor cores.  Built for the shape the reference trains (src/main.cpp:203-213, src/NeRFExecutor.h:507-514):
 * LeRF(geo_feat_dim_le 32, num_layers_le 2, hidden_dim_le 256, lang_embed_dim 512, input_ch_le 16 levels x 8 features = 128), every
 * layer bias-free (src/LeRF.cpp:12,15); other shapes return NRF_ERR_UNSUPPORTED.  enc_f16 [N,128] fp16 is the output of
 * nrf_hash_encode_fwd on the language grid (n_features 8); keep u8 [N] (nullable) its keep mask.
 *
 *   nrf_lerf_pack              weights (torch Linear layout [out,in] fp32) -> operand blob (nrf_lerf_packed_bytes, 128-byte aligned)
 *   nrf_lerf_fwd               raw_le [N, 513] fp32 = [normalize(e, eps 1e-8) (512) | sigma_le], sigma_le := 0 where keep == 0
 *                              (what LeRF::forward + RunLENetwork return; the compatibility entry)
 *   nrf_lerf_sigma_fwd         raw4 [N,4] fp32 = [0,0,0,sigma_le]: the coarse pass of LeRFRenderer::RenderRays only needs the density
 *                              (src/LeRFRenderer.cpp:133-139); raw4 is what nrf_composite_fwd (raw_stride 4) consumes
 *   nrf_lerf_hidden_fwd        the fine pass without the [N,512] embedding: raw4 as above, `hidden` = the last hidden layer h2 as fp16
 *                              tile records (nrf_lerf_hidden_bytes(n) bytes, 128-byte aligned), q [N] fp32 = |W_e1 h2|^2
 *   nrf_lerf_render_embedding  weights [R,S] fp32 (WeightsLE from nrf_composite_fwd on raw4) + hidden + q ->
 *                              rendered [R,512] = normalize(sum_s w_s e_s / max(|e_s|, 1e-8), eps 1e-8), evaluated as
 *                              normalize(W_e1 sum_s (w_s / |e_s|) h2_s); hsum [R,256] fp32 is caller-owned workspace
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct nrf_lerf_shape {
	int32_t geo_feat_dim;     /* 32  */
	int32_t num_layers;       /* 2   */
	int32_t hidden_dim;       /* 256 */
	int32_t lang_embed_dim;   /* 512 */
	int32_t input_ch;         /* 128 */
} nrf_lerf_shape;

typedef struct nrf_lerf_weights {   /* device pointers, fp32 row-major [out, in]; names as registered by src/LeRF.cpp:17-25 */
	const float* sigma_w0;    /* <name>_sigma_le_net_0.weight [256, 128] */
	const float* sigma_w1;    /* <name>_sigma_le_net_1.weight [33, 256]: row 0 sigma_le, rows 1..32 geo_feat_le */
	const float* le_w0;       /* <name>_le_net_0.weight [256, 160]: columns [geo_feat_le 32 | inputs_le 128] */
	const float* le_w1;       /* <name>_le_net_1.weight [512, 256] */
} nrf_lerf_weights;

int64_t nrf_lerf_packed_bytes(const nrf_lerf_shape* shape);
int64_t nrf_lerf_hidden_bytes(const nrf_lerf_shape* shape, int64_t n);
int nrf_lerf_pack(const nrf_lerf_shape* shape, const nrf_lerf_weights* weights, void* packed, nrf_stream stream);
int nrf_lerf_fwd(const nrf_lerf_shape* shape, const void* packed, const void* enc_f16, const uint8_t* keep, int64_t n, float* raw_le,
                 nrf_stream stream);
int nrf_lerf_sigma_fwd(const nrf_lerf_shape* shape, const void* packed, const void* enc_f16, const uint8_t* keep, int64_t n, float* raw4,
                       nrf_stream stream);
int nrf_lerf_hidden_fwd(const nrf_lerf_shape* shape, const void* packed, const void* enc_f16, const uint8_t* keep, int64_t n, float* raw4,
                        void* hidden, float* q, nrf_stream stream);
int nrf_lerf_render_embedding(const nrf_lerf_shape* shape, const void* packed, const float* weights, const void* hidden, const float* q,
                              int64_t n_rays, int32_t n_samples, float* hsum, float* rendered, nrf_stream stream);

/* Training of the language field — replaces LibTorch autograd behind LeRFImpl::forward (src/LeRF.cpp:78-110), RenderCLIPEmbedding
 * (src/LeRFRenderer.h:45-54) inside RawToLEOutputs (src/LeRFRenderer.cpp:27-82) and the language loss (src/NeRFExecutor.h:957-983).
 * bf16 operands, fp32 accumulation; the [N,512] embedding is formed neither forward nor backward.  One fine-pass batch of n = n_rays *
 * n_samples rows (the coarse pass is never differentiated, SURVEY §9-Q3) goes through, in order:
 *   nrf_lerf_fwd_train               enc -> raw4 [N,4] = [0,0,0,sigma_le], q [N] = |W_e1 h2|^2, `saved` (nrf_lerf_train_saved_bytes(n) bytes,
 *                                    128-byte aligned): per 128-row tile the bf16 records [x | geo], h1, h2 and the ReLU mask of h1
 *   nrf_composite_fwd                (existing) raw4 -> comp_weights [R,S]
 *   nrf_lerf_render_embedding_train  -> hsum [R,256], rendered [R,512], enorm [R] = |W_e1 hsum|
 *   nrf_lerf_bwd_rays                d loss / d rendered — either grad_rendered [R,512] (any loss; target NULL) or the reference's loss
 *                                    formed here from target [R,512] (huber delta 1.25 summed over channels, mean over rays; loss_out[0] +=
 *                                    loss, grad_rendered NULL) — times grad_scale -> grad_le_w1 [512,256] += dE Hs^T, dw_out [R,S] =
 *                                    d loss / d comp_weights; per-ray / per-row coefficients stay in `workspace`
 *                                    (nrf_lerf_bwd_workspace_bytes(n, n_rays) bytes, 256-byte aligned, caller-owned, reused by the next entry)
 *   nrf_composite_bwd                (existing) g_weights = dw_out -> d_raw4 [N,4]
 *   nrf_lerf_bwd_rows                gradient chain + weight gradients: grads->{sigma_w0, sigma_w1, le_w0, le_w1} += (fp32, the shapes
 *                                    of `weights`; the struct's pointers are written through), d_enc_bf16 [N,128] bf16 = d loss / d enc, the
 *                                    layout nrf_hash_encode_bwd (NRF_GRAD_BF16) reads.  `packed` must be the blob of the same `weights`. */
int64_t nrf_lerf_train_saved_bytes(const nrf_lerf_shape* shape, int64_t n);
int64_t nrf_lerf_bwd_workspace_bytes(const nrf_lerf_shape* shape, int64_t n, int64_t n_rays);
int nrf_lerf_fwd_train(const nrf_lerf_shape* shape, const void* packed, const void* enc_f16, const uint8_t* keep, int64_t n, float* raw4,
                       void* saved, float* q, nrf_stream stream);
int nrf_lerf_render_embedding_train(const nrf_lerf_shape* shape, const void* packed, const float* weights, const void* saved,
                                    const float* q, int64_t n_rays, int32_t n_samples, float* hsum, float* rendered, float* enorm,
                                    nrf_stream stream);
int nrf_lerf_bwd_rays(const nrf_lerf_shape* shape, const nrf_lerf_weights* weights, const void* saved, const float* q,
                      const float* comp_weights, const float* hsum, const float* rendered, const float* enorm, const float* target,
                      const float* grad_rendered, int64_t n_rays, int32_t n_samples, float grad_scale, float* loss_out,
                      float* grad_le_w1, void* workspace, float* dw_out, nrf_stream stream);
int nrf_lerf_bwd_rows(const nrf_lerf_shape* shape, const void* packed, const nrf_lerf_weights* weights, const void* saved,
                      const uint8_t* keep, const float* d_raw4, int64_t n, int32_t n_samples, void* workspace,
                      const nrf_lerf_weights* grads, void* d_enc_bf16, nrf_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* NERFPP_B200_H */
