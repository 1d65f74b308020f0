// HashNeRFTrainGraph (see train_graph.h).  Every arithmetic step is a C-ABI call; torch supplies memory, the stream and the graph capture.
#include "train_graph.h"

#include <c10/cuda/CUDAStream.h>

using torch::Tensor;

namespace {
Tensor F32(std::initializer_list<int64_t> shape, const torch::Device& d) { return torch::empty(shape, torch::TensorOptions().dtype(torch::kFloat32).device(d)); }
}

HashNeRFTrainGraph::HashNeRFTrainGraph(CuHashEmbedder embed, CuSHEncoder embeddirs, NeRFSmall model, Tensor bounding_box, int n_samples,
	int n_importance, float learning_rate, int lrate_decay, int64_t n_rays)
	: Embed(embed), EmbedDirs(embeddirs), Model(model), S(n_samples), N(n_importance), Lr0(learning_rate), LrateDecay(lrate_decay), R(n_rays)
{
	TORCH_CHECK(Model->Fused() && Embed->GetOutputDims() == Model->GetInputCh() && EmbedDirs->GetDegree() * EmbedDirs->GetDegree() == Model->GetInputChViews(),
		"HashNeRFTrainGraph: built for the fused NeRFSmall shape (32 hash channels + SH degree 4)");
	TORCH_CHECK(n_importance > 0 && n_rays > 0 && (S + N) < 32768, "HashNeRFTrainGraph: n_importance > 0, n_rays > 0");
	TORCH_CHECK(Embed->Embeddings.is_cuda(), "HashNeRFTrainGraph: the modules must be on the GPU (there is no CPU path)");
	Box = nrfhost::HostBox(bounding_box);
	const torch::Device dev = Embed->Embeddings.device();
	c10::cuda::CUDAGuard guard(dev);
	torch::NoGradGuard no_grad;

	// ---- one flat parameter vector [Embeddings | sigma_net_0, sigma_net_1, color_net_0, color_net_1, color_net_2]; the modules' parameters become views
	std::vector<Tensor> w = Model->Weights();
	NTableAll = Embed->Embeddings.numel();
	NMlp = 0;
	for (const Tensor& t : w) NMlp += t.numel();
	{
		// scalars the kernels can reach: level offsets are in scalars (src/CuHashEmbedder.cu:55,150), so only a prefix of the [L*2^T, F] parameter
		Tensor idx = Embed->FeatLocalIdx.to(torch::kCPU, torch::kInt64), size = Embed->FeatLocalSize.to(torch::kCPU, torch::kInt64);
		NTableUsed = 0;
		for (int64_t l = 0; l < idx.numel(); l++)
			NTableUsed = std::max<int64_t>(NTableUsed, idx[l].item<int64_t>() + size[l].item<int64_t>() * Embed->NFeaturesPerLevel);
		NTableUsed = std::min<int64_t>((NTableUsed + 3) / 4 * 4, NTableAll);
	}
	P = torch::empty({NTableAll + NMlp}, torch::TensorOptions().dtype(torch::kFloat32).device(dev));
	P.narrow(0, 0, NTableAll).copy_(Embed->Embeddings.detach().reshape({-1}));
	Embed->Embeddings.set_data(P.narrow(0, 0, NTableAll).view(Embed->Embeddings.sizes()));
	int64_t off = NTableAll;
	for (Tensor& t : w) {
		P.narrow(0, off, t.numel()).copy_(t.detach().reshape({-1}));
		t.set_data(P.narrow(0, off, t.numel()).view(t.sizes()));
		off += t.numel();
	}
	G = torch::zeros_like(P);
	M = torch::zeros_like(P);
	V = torch::zeros_like(P);
	Shadow = torch::empty({P.numel()}, torch::TensorOptions().dtype(torch::kFloat16).device(dev));
	nrfhost::Check(nrf_table_to_half(P.data_ptr<float>(), Shadow.data_ptr(), NTableAll, nrfhost::Stream()), "nrf_table_to_half");
	const nrf_mlp_small_shape shape = Model->Shape();
	Packed = torch::empty({nrf_mlp_small_packed_bytes(&shape)}, torch::TensorOptions().dtype(torch::kUInt8).device(dev));
	nrfhost::Check(nrf_mlp_small_pack(&shape, P.data_ptr<float>() + NTableAll, Packed.data_ptr(), nrfhost::Stream()), "nrf_mlp_small_pack");
	Sched = torch::zeros({4}, torch::TensorOptions().dtype(torch::kInt32).device(dev));
	Loss = torch::zeros({1}, torch::TensorOptions().dtype(torch::kFloat32).device(dev));
	TVals = torch::linspace(0.0, 1.0, S, torch::TensorOptions().dtype(torch::kFloat32)).to(dev);      // src/NeRFRenderer.h:393
	U = torch::linspace(0.0, 1.0, N, torch::TensorOptions().dtype(torch::kFloat32)).to(dev);          // src/Sampler.h:20
	InO = F32({R, 3}, dev); InD = F32({R, 3}, dev); InT = F32({R, 3}, dev);
	InO.zero_(); InT.fill_(0.5f);
	InD.zero_(); InD.select(1, 2).fill_(-1.f);
	InO.select(1, 2).fill_(4.f);

	// ---- warm-up outside the capture (function attributes, level scales, allocator pools): render + loss + backward only, gradient discarded;
	// then the capture itself, both on a side stream
	c10::cuda::CUDAStream side = c10::cuda::getStreamFromPool(false, dev.index());
	C10_CUDA_CHECK(cudaStreamSynchronize(c10::cuda::getCurrentCUDAStream(dev.index()).stream()));
	{
		c10::cuda::CUDAStreamGuard sg(side);
		Enqueue(false);
		G.zero_();
		Keep.clear();
		C10_CUDA_CHECK(cudaStreamSynchronize(side.stream()));
		const int64_t before = nrf_launch_count();
		Graph.capture_begin();
		Enqueue(true);
		Graph.capture_end();
		Kernels = static_cast<int>(nrf_launch_count() - before);
		C10_CUDA_CHECK(cudaStreamSynchronize(side.stream()));
	}
}

void HashNeRFTrainGraph::Enqueue(bool with_optimizer)
{
	const torch::Device dev = P.device();
	const nrf_stream st = nrfhost::Stream();
	const nrf_mlp_small_shape shape = Model->Shape();
	nrf_hash_grid grid = Embed->Grid();
	const int64_t nc = R * S, nf = R * (S + N);
	const int sf = S + N;
	const auto u8 = torch::TensorOptions().dtype(torch::kUInt8).device(dev);
	float* const g_table = G.data_ptr<float>();
	float* const g_mlp = G.data_ptr<float>() + NTableAll;
	const void* table16 = Shadow.data_ptr();

	Tensor ray_batch = F32({R, 11}, dev), z = F32({R, S}, dev), ray_sh = F32({R, 16}, dev);
	nrfhost::Check(nrf_ray_setup(InO.data_ptr<float>(), InD.data_ptr<float>(), R, Box.data(), 0.f, TVals.data_ptr<float>(), S, 0, EmbedDirs->GetDegree(),
		ray_batch.data_ptr<float>(), z.data_ptr<float>(), ray_sh.data_ptr<float>(), Loss.data_ptr<float>(), st), "nrf_ray_setup");
	// coarse pass (inference: it never receives a gradient, src/NeRFRenderer.h:422-431)
	Tensor enc_c = torch::empty({nc, 32}, torch::TensorOptions().dtype(torch::kFloat16).device(dev)), keep_c = torch::empty({nc}, u8), raw_c = F32({R, S, 4}, dev);
	nrfhost::Check(nrf_hash_encode_rays_fwd(&grid, table16, ray_batch.data_ptr<float>(), 11, z.data_ptr<float>(), R, S, 1, keep_c.data_ptr<uint8_t>(),
		enc_c.data_ptr(), NRF_ENC_F16, nullptr, nullptr, nullptr, 0, st), "nrf_hash_encode_rays_fwd");
	nrfhost::Check(nrf_mlp_small_fwd(&shape, Packed.data_ptr(), NRF_MLP_IN_ENC16_RAYDIRS, enc_c.data_ptr(), ray_sh.data_ptr<float>(), S, keep_c.data_ptr<uint8_t>(), nc,
		raw_c.data_ptr<float>(), st), "nrf_mlp_small_fwd");
	Tensor rgb_c = F32({R, 3}, dev), depth = F32({R}, dev), disp = F32({R}, dev), acc = F32({R}, dev), w_c = F32({R, S}, dev);
	nrfhost::Check(nrf_composite_fwd(raw_c.data_ptr<float>(), 4, z.data_ptr<float>(), InD.data_ptr<float>(), nullptr, 0.f, 0, R, S, rgb_c.data_ptr<float>(),
		depth.data_ptr<float>(), disp.data_ptr<float>(), acc.data_ptr<float>(), w_c.data_ptr<float>(), st), "nrf_composite_fwd");
	// importance samples; the merged list contains the coarse samples bit for bit, so their encoding rows are copied, not gathered again, and
	// (one network for both passes, src/NeRFRenderer.h:422,447) their raw rows are the coarse pass's: the fine forward evaluates the N new samples
	Tensor z_f = F32({R, sf}, dev), perm = torch::empty({R, sf}, torch::TensorOptions().dtype(torch::kInt16).device(dev));
	Tensor enc = torch::empty({nf, 32}, torch::TensorOptions().dtype(torch::kFloat16).device(dev)), keep = torch::empty({nf}, u8), raw = F32({R, sf, 4}, dev);
	nrfhost::Check(nrf_sample_pdf_merge_rows(z.data_ptr<float>(), w_c.data_ptr<float>(), U.data_ptr<float>(), 0, R, S, N, nullptr, z_f.data_ptr<float>(),
		perm.data_ptr<int16_t>(), raw_c.data_ptr<float>(), raw.data_ptr<float>(), st), "nrf_sample_pdf_merge_rows");
	nrfhost::Check(nrf_hash_encode_rays_fwd(&grid, table16, ray_batch.data_ptr<float>(), 11, z_f.data_ptr<float>(), R, sf, 1, keep.data_ptr<uint8_t>(), enc.data_ptr(),
		NRF_ENC_F16, perm.data_ptr<int16_t>(), enc_c.data_ptr(), keep_c.data_ptr<uint8_t>(), S, st), "nrf_hash_encode_rays_fwd");
	nrfhost::Check(nrf_mlp_small_fwd_importance(&shape, Packed.data_ptr(), NRF_MLP_IN_ENC16_RAYDIRS, enc.data_ptr(), ray_sh.data_ptr<float>(), keep.data_ptr<uint8_t>(),
		perm.data_ptr<int16_t>(), R, N, sf, raw.data_ptr<float>(), st), "nrf_mlp_small_fwd_importance");
	// RawToOutputs of the fine pass + huber_loss + their backward (src/NeRFRenderer.h:447-448, src/NeRFExecutor.h:883-890, 923): one launch
	Rgb = F32({R, 3}, dev);
	Tensor d_raw = F32({R, sf, 4}, dev);
	nrfhost::Check(nrf_composite_huber_bwd(raw.data_ptr<float>(), 4, z_f.data_ptr<float>(), InD.data_ptr<float>(), nullptr, 0.f, 0, R, sf, InT.data_ptr<float>(), 1.f, 1.f,
		Loss.data_ptr<float>(), Rgb.data_ptr<float>(), d_raw.data_ptr<float>(), st), "nrf_composite_huber_bwd");
	Tensor g_enc = torch::empty({nf, 32}, torch::TensorOptions().dtype(torch::kBFloat16).device(dev));
	nrfhost::Check(nrf_mlp_small_bwd(&shape, Packed.data_ptr(), NRF_MLP_IN_ENC16_RAYDIRS, enc.data_ptr(), ray_sh.data_ptr<float>(), sf, keep.data_ptr<uint8_t>(), nf,
		d_raw.data_ptr<float>(), g_enc.data_ptr(), g_mlp, st), "nrf_mlp_small_bwd");
	nrfhost::Check(nrf_hash_encode_rays_bwd(&grid, ray_batch.data_ptr<float>(), 11, z_f.data_ptr<float>(), R, sf, 1, g_enc.data_ptr(), NRF_GRAD_BF16, g_table, st),
		"nrf_hash_encode_rays_bwd");
	Keep = {ray_batch, z, ray_sh, enc_c, keep_c, raw_c, rgb_c, depth, disp, acc, w_c, z_f, perm, enc, keep, raw, d_raw, g_enc};
	if (!with_optimizer) return;
	// Optimizer->step() + the decayed rate (src/NeRFExecutor.h:539, 986-996): schedule record advanced on the device, Adam over the reachable table
	// prefix (+ fp16 shadow + gradient clear) and over the weights, re-pack
	nrfhost::Check(nrf_adam_schedule_advance(Sched.data_ptr(), Lr0, 0.1f, float(LrateDecay) * 1000.f, 0.9f, 0.99f, st), "nrf_adam_schedule_advance");
	nrfhost::Check(nrf_adam_step_scheduled(P.data_ptr<float>(), g_table, M.data_ptr<float>(), V.data_ptr<float>(), NTableUsed, Sched.data_ptr(), 0.9f, 0.99f, 1e-15f,
		1.f, 1, Shadow.data_ptr(), st), "nrf_adam_step_scheduled");
	nrfhost::Check(nrf_adam_step_scheduled(P.data_ptr<float>() + NTableAll, g_mlp, M.data_ptr<float>() + NTableAll, V.data_ptr<float>() + NTableAll, NMlp, Sched.data_ptr(),
		0.9f, 0.99f, 1e-15f, 1.f, 1, static_cast<at::Half*>(Shadow.data_ptr()) + NTableAll, st), "nrf_adam_step_scheduled");
	nrfhost::Check(nrf_mlp_small_pack(&shape, P.data_ptr<float>() + NTableAll, Packed.data_ptr(), st), "nrf_mlp_small_pack");
}

Tensor HashNeRFTrainGraph::Step(const Tensor& rays_o, const Tensor& rays_d, const Tensor& target)
{
	TORCH_CHECK(rays_o.size(0) == R && rays_d.size(0) == R && target.size(0) == R, "HashNeRFTrainGraph: captured for ", R, " rays");
	c10::cuda::CUDAGuard guard(P.device());
	torch::NoGradGuard no_grad;
	InO.copy_(rays_o, /*non_blocking=*/true);
	InD.copy_(rays_d, true);
	InT.copy_(target, true);
	Graph.replay();
	Steps++;
	// the data changed behind autograd's back: modules caching derived copies (fp16 table shadow, packed weights) must see it
	Embed->Embeddings.unsafeGetTensorImpl()->bump_version();
	for (Tensor& t : Model->Weights()) t.unsafeGetTensorImpl()->bump_version();
	return Loss;
}
