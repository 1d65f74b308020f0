// NeRFExecutor::Train's loop body for NeRFRenderer<CuHashEmbedder, CuSHEncoder, NeRFSmall> as ONE CUDA-graph replay on the C++ surface.
//
// The reference's iteration (src/NeRFExecutor.h:868-890, 923, 986-996) is
//     Optimizer->zero_grad(); Render(rays) -> huber_loss(RGBMap, target) -> loss.backward(); Optimizer->step(); set_lr(decayed)
// which, on the drop-in classes, is ~60 kernel launches behind ATen / autograd bookkeeping (1.2 ms per 4096-ray step, of which 0.8 ms is kernel
// time).  HashNeRFTrainGraph runs the SAME step — the same C-ABI kernels in the same order as the autograd path issues them — as one captured
// graph of 14 kernel nodes:
//     ray setup -> [hash encode -> NeRFSmall] coarse -> RawToOutputs -> SamplePDF + merge -> [hash encode -> NeRFSmall] fine ->
//     RawToOutputs + huber + RawToOutputs backward (one kernel) -> NeRFSmall backward -> hash scatter -> Adam (+ fp16 shadow, gradient clear,
//     LR schedule on the device) -> weight re-pack
// By default the parity configuration of the benchmark (ThinRay, Perturb 0, no raw noise, no stochastic preconditioning, coarse pass not
// differentiated — SURVEY §9-Q3/Q4).  The reference's shipped configuration (src/main.cpp:187 thin_ray = false, SH degree 8, RawNoiseStd and
// StochasticPreconditioningAlpha from the caller's schedule, src/NeRFExecutor.h:411-412) runs through the Step overload that takes the cone
// angle and the step's two amplitudes: the jittered points are generated inside the hash kernels (nrf_hash_encode_rays_jitter_fwd / _bwd), the
// fine pass evaluates all S+N samples (a jittered coarse sample is re-jittered with fresh draws), and the variates are the SAME torch::rand /
// torch::randn calls the autograd path issues (chunk by chunk, as BatchifyRays would), captured into the graph: torch's CUDA generator
// advances its offset per replay, so with the same seed the graph consumes exactly the autograd loop's draws.  Noise and preconditioning are
// drawn only when their amplitude is > 0, as in the reference: each of the (at most 4) combinations is its own graph, captured the first
// time a step needs it; all of them share one memory pool.  Any SH degree 1..8: at a view width other than 16 the colour net's view term
// enters the fused kernels per ray (nrf_mlp_small_view_bias_fwd / _bwd, NRF_MLP_IN_ENC16_RAYBIAS).
//
// The modules stay the owners of their parameters: at construction the embedder's Embeddings and the five NeRFSmall weights are re-pointed
// (Tensor::set_data) at slices of ONE flat fp32 vector, so parameters(), named_parameters(), torch::save / torch::load archives and the
// autograd path keep working on the same storage, while the step needs one gradient buffer and two Adam launches (table prefix the kernels can
// reach, then the 9 344 weights).  Adam moments live here; they are exposed for optimiser checkpoints (ExpAvg / ExpAvgSq / StepCount).
#pragma once
#include <ATen/cuda/CUDAGraph.h>

#include "embedders.h"
#include "models.h"

class HashNeRFTrainGraph {
public:
	/// thin_ray false: TangentScatter jitter in both passes (the cone angle comes with every Step).  chunk (0 = n_rays): the ray count of one
	/// RenderRays call of the autograd path (BatchifyRays, src/NeRFRenderer.h:465-525), which sets the layout of the variates drawn per step.
	HashNeRFTrainGraph(CuHashEmbedder embed, CuSHEncoder embeddirs, NeRFSmall model, torch::Tensor bounding_box, int n_samples, int n_importance,
		float learning_rate, int lrate_decay, int64_t n_rays, bool thin_ray = true, int64_t chunk = 0);
	/// one optimisation step on rays_o / rays_d [n_rays,3] and target [n_rays,3] (device or pinned host tensors); returns the loss (device scalar,
	/// overwritten by the next step).  Thin rays, no noise, no preconditioning.
	torch::Tensor Step(const torch::Tensor& rays_o, const torch::Tensor& rays_d, const torch::Tensor& target);
	/// the same with the shipped configuration's per-step inputs: cone_angle (scalar or [n_rays], ignored for thin rays) and the amplitudes the
	/// caller's FillRenderParams(i) computes (src/NeRFExecutor.h:411-412); > 0 switches the stage on
	torch::Tensor Step(const torch::Tensor& rays_o, const torch::Tensor& rays_d, const torch::Tensor& target, const torch::Tensor& cone_angle,
		float raw_noise_std, float sp_alpha);
	int64_t StepCount() const { return Steps; }
	/// library kernels per step of the graph the last step replayed (torch's RNG and scaling kernels not counted)
	int KernelsPerStep() const { return Kernels[Last]; }
	bool ThinRay() const { return Thin; }
	torch::Tensor ExpAvg() const { return M; }
	torch::Tensor ExpAvgSq() const { return V; }
	torch::Tensor RGB() const { return Rgb; }        ///< RGBMap of the last step [n_rays,3]

private:
	void Enqueue(bool with_optimizer, int stage);     ///< the step's kernels on the current stream (stage bit 0: noise, bit 1: preconditioning)
	void Capture(int stage);                          ///< warm-up + capture of one stage's graph; consumes no draws of the CUDA generator
	CuHashEmbedder Embed = nullptr;
	CuSHEncoder EmbedDirs = nullptr;
	NeRFSmall Model = nullptr;
	std::array<float, 6> Box{};
	int S, N, Deg;
	bool Thin, RayBias;
	int64_t Chunk;
	float Lr0;
	int LrateDecay;
	int64_t R, NTableAll, NTableUsed, NMlp, Steps = 0;
	torch::Tensor P, G, M, V, Shadow, Packed, Sched, Loss, TVals, U, InO, InD, InT, Rgb;
	torch::Tensor InCone, NoiseStd, SpAlpha;          ///< per-step inputs of the shipped configuration: [n_rays] cone angles, two device scalars
	std::array<std::unique_ptr<at::cuda::CUDAGraph>, 4> Graphs;   ///< one per stage, captured on first use
	std::array<std::vector<torch::Tensor>, 4> Keep;  ///< intermediates of each captured step (their storage belongs to the graphs' pool)
	std::array<int, 4> Kernels{};
	int Last = 0;
	at::cuda::MempoolId_t Pool;
};
