// pybind11 front-end of the C++ drop-in layer (nerfpp_b200/host/*.h) -> nerfpp_b200/lib/nerfpp_b200_torch*.so.
// It exposes the SAME call surface as oracle/ref_bindings.cpp exposes for the reference, so tests/test_gpu_host.py drives
// both modules with identical code and compares results; bench.py uses train_steps() as the C++ training loop
// (the lines of NeRFExecutor::Train that touch this path, src/NeRFExecutor.h:539,868,876-890,923,986,992-996).
#include <torch/extension.h>
#include <chrono>

#include "renderer.h"
#include "lerf.h"
#include "fused_adam.h"
#include "train_graph.h"

namespace py = pybind11;
using torch::Tensor;

template <class E, class D, class N>
struct OpenRenderer : public NeRFRenderer<E, D, N> {
	using Base = NeRFRenderer<E, D, N>;
	using Base::Base;
	using Base::RunNetwork;
	using Base::RawToOutputs;
	using Base::NeRF;
	using Base::EmbedFn;
	using Base::EmbeddirsFn;
};

static py::dict ToDict(const NeRFRendererOutputs& o)
{
	py::dict d;
	d["rgb"] = o.RGBMap; d["disp"] = o.DispMap; d["acc"] = o.AccMap; d["weights"] = o.Weights; d["depth"] = o.DepthMap;
	return d;
}

static NeRFRenderParams Params(int n_samples, int n_importance, int chunk, bool white, bool use_viewdirs, Tensor bbox, bool thin_ray,
	float raw_noise_std, float sp_alpha)
{
	NeRFRenderParams p;
	p.NSamples = n_samples; p.NImportance = n_importance; p.Chunk = chunk; p.ReturnRaw = false; p.LinDisp = false; p.Perturb = 0.f;
	p.WhiteBkgr = white; p.RawNoiseStd = raw_noise_std; p.Ndc = false; p.UseViewdirs = use_viewdirs; p.ReturnWeights = true;
	p.ThinRay = thin_ray; p.BoundingBox = bbox; p.StochasticPreconditioningAlpha = sp_alpha;
	return p;
}

template <class E, class D, class N>
struct Pipeline {
	E embed{nullptr};
	D embeddirs{nullptr};
	N model{nullptr};
	std::unique_ptr<OpenRenderer<E, D, N>> renderer;
	std::unique_ptr<torch::optim::Adam> opt;
	Tensor bbox;
	int global_step = 0;

	void Finish()
	{
		embed->to(torch::kCUDA); embeddirs->to(torch::kCUDA); model->to(torch::kCUDA);
		renderer = std::make_unique<OpenRenderer<E, D, N>>(embed, embeddirs, model);
	}
	std::vector<Tensor> EmbedParams() { return embed->parameters(); }
	std::vector<Tensor> ModelParams() { return model->parameters(); }
	std::vector<std::string> ModelParamNames() { std::vector<std::string> r; for (auto& p : model->named_parameters()) r.push_back(p.key()); return r; }
	std::vector<std::string> EmbedParamNames() { std::vector<std::string> r; for (auto& p : embed->named_parameters()) r.push_back(p.key()); return r; }
	std::vector<std::string> EmbedBufferNames() { std::vector<std::string> r; for (auto& p : embed->named_buffers()) r.push_back(p.key()); return r; }
	std::vector<Tensor> EmbedBuffers() { return embed->buffers(); }
	void InitModel() { Trainable::Initialize(model); }
	int OutputDims() { return embed->GetOutputDims(); }
	std::pair<Tensor, Tensor> Embed(Tensor x) { return embed->forward(x); }
	Tensor EmbedDirs(Tensor d) { return embeddirs->forward(d).first; }
	Tensor Model(Tensor x) { return model->forward(x); }
	Tensor RunNetwork(Tensor pts, Tensor viewdirs) { return renderer->RunNetwork(pts, viewdirs, renderer->NeRF, renderer->EmbedFn, renderer->EmbeddirsFn); }
	py::dict RawToOutputs(Tensor raw, Tensor z, Tensor rays_d, float noise, bool white) { return ToDict(renderer->RawToOutputs(raw, Tensor(), z, rays_d, noise, white)); }
	py::dict RenderRays(Tensor ray_batch, int n_samples, int n_importance, bool white, bool return_raw)
	{
		auto r = renderer->RenderRays(ray_batch, Tensor(), n_samples, return_raw, false, 0.f, n_importance, white, 0.f, 0.f, bbox, true);
		py::dict d = ToDict(r.Outputs);
		if (return_raw) d["raw"] = r.Raw;
		return d;
	}
	py::dict Render(Tensor rays_o, Tensor rays_d, int n_samples, int n_importance, int chunk, bool white, bool use_viewdirs)
	{
		auto p = Params(n_samples, n_importance, chunk, white, use_viewdirs, bbox, true, 0.f, 0.f);
		auto r = renderer->Render(0, 0, Tensor(), p, {rays_o, rays_d, Tensor()}, Tensor(), Tensor());
		py::dict d = ToDict(r.Outputs);
		d["near"] = r.Near; d["far"] = r.Far;
		return d;
	}
	// the as-shipped configuration (src/main.cpp:187: thin_ray = false, raw noise and stochastic preconditioning on)
	py::dict RenderShipped(Tensor rays_o, Tensor rays_d, Tensor cone_angle, int n_samples, int n_importance, int chunk, float raw_noise_std, float sp_alpha)
	{
		auto p = Params(n_samples, n_importance, chunk, false, true, bbox, false, raw_noise_std, sp_alpha);
		auto r = renderer->Render(0, 0, Tensor(), p, {rays_o, rays_d, cone_angle}, Tensor(), Tensor());
		return ToDict(r.Outputs);
	}
	py::dict RenderImage(int h, int w, Tensor k, Tensor c2w, int n_samples, int n_importance, int chunk, bool white, bool use_viewdirs)
	{
		torch::NoGradGuard ng;
		auto p = Params(n_samples, n_importance, chunk, white, use_viewdirs, bbox, true, 0.f, 0.f);
		auto r = renderer->Render(h, w, k, p, {Tensor(), Tensor(), Tensor()}, c2w, Tensor());
		py::dict d = ToDict(r.Outputs);
		d["near"] = r.Near; d["far"] = r.Far;
		return d;
	}
	bool fused_adam = false;   ///< FusedAdam (one sm_100a kernel per parameter) instead of torch::optim::Adam; chosen before the first step
	void UseFusedAdam(bool on) { TORCH_CHECK(!opt, "choose the optimiser before the first training step"); fused_adam = on; }
	bool train_graph = false;  ///< HashNeRFTrainGraph: the whole iteration as one CUDA-graph replay (HashNeRF instantiation only)
	std::unique_ptr<HashNeRFTrainGraph> graph;
	void UseTrainGraph(bool on) { TORCH_CHECK(!opt && !graph, "choose the training path before the first training step"); train_graph = on; }
	std::pair<std::vector<double>, std::vector<float>> TrainSteps(Tensor rays_o, Tensor rays_d, Tensor target, int n_steps, int n_samples,
		int n_importance, int chunk, bool use_viewdirs, float lr, int lrate_decay)
	{
		if constexpr (std::is_same_v<N, NeRFSmall>) {
			if (train_graph) {
				// NeRFExecutor::Train's iteration as one graph replay; loss.item() every step like the reference's loop
				if (!graph) graph = std::make_unique<HashNeRFTrainGraph>(embed, embeddirs, model, bbox, n_samples, n_importance, lr, lrate_decay, rays_o.size(0));
				std::vector<double> secs; std::vector<float> losses;
				for (int i = 0; i < n_steps; i++) {
					auto t0 = std::chrono::steady_clock::now();
					const float lv = graph->Step(rays_o, rays_d, target).template item<float>();
					secs.push_back(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
					losses.push_back(lv);
				}
				return {secs, losses};
			}
		}
		if (!opt) {
			std::vector<Tensor> gv;
			for (auto& p : embed->parameters()) gv.push_back(p);
			for (auto& p : model->parameters()) gv.push_back(p);
			const auto options = torch::optim::AdamOptions(lr).eps(1e-15).betas(std::make_tuple(0.9, 0.99));
			if (fused_adam) opt = std::make_unique<FusedAdam>(gv, options);
			else opt = std::make_unique<torch::optim::Adam>(gv, options);
			global_step = 0;
		}
		std::vector<double> secs; std::vector<float> losses;
		auto p = Params(n_samples, n_importance, chunk, false, use_viewdirs, bbox, true, 0.f, 0.f);
		for (int i = 0; i < n_steps; i++) {
			auto t0 = std::chrono::steady_clock::now();
			opt->zero_grad();
			auto r = renderer->Render(0, 0, Tensor(), p, {rays_o, rays_d, Tensor()}, Tensor(), Tensor());
			auto loss = torch::nn::functional::huber_loss(r.Outputs.RGBMap, target.detach());
			loss.backward();
			opt->step();
			const float new_lr = lr * powf(0.1f, float(global_step) / (lrate_decay * 1000));
			for (auto& g : opt->param_groups()) g.options().set_lr(new_lr);
			global_step++;
			const float lv = loss.template item<float>();
			secs.push_back(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
			losses.push_back(lv);
		}
		return {secs, losses};
	}
	/// NeRFExecutor::Train's loop in the reference's shipped configuration (src/main.cpp:187 thin_ray = false; the per-step RawNoiseStd and
	/// StochasticPreconditioningAlpha of FillRenderParams(i), src/NeRFExecutor.h:411-412, given as schedules): the graph of train_graph.h, or the
	/// autograd loop over Render when use_train_graph(False)
	std::pair<std::vector<double>, std::vector<float>> TrainStepsShipped(Tensor rays_o, Tensor rays_d, Tensor target, Tensor cone, int n_steps,
		int n_samples, int n_importance, int chunk, float lr, int lrate_decay, std::vector<float> noise_std, std::vector<float> sp_alpha)
	{
		TORCH_CHECK(int(noise_std.size()) >= n_steps && int(sp_alpha.size()) >= n_steps, "train_steps_shipped: one noise / alpha value per step");
		if constexpr (std::is_same_v<N, NeRFSmall>) {
			if (train_graph) {
				if (!graph)
					graph = std::make_unique<HashNeRFTrainGraph>(embed, embeddirs, model, bbox, n_samples, n_importance, lr, lrate_decay, rays_o.size(0), false, chunk);
				TORCH_CHECK(!graph->ThinRay(), "train_steps_shipped: this pipe's training graph was built for thin rays (train_steps)");
				std::vector<double> secs; std::vector<float> losses;
				for (int i = 0; i < n_steps; i++) {
					auto t0 = std::chrono::steady_clock::now();
					const float lv = graph->Step(rays_o, rays_d, target, cone, noise_std[i], sp_alpha[i]).template item<float>();
					secs.push_back(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
					losses.push_back(lv);
				}
				return {secs, losses};
			}
		}
		if (!opt) {
			std::vector<Tensor> gv;
			for (auto& p : embed->parameters()) gv.push_back(p);
			for (auto& p : model->parameters()) gv.push_back(p);
			const auto options = torch::optim::AdamOptions(lr).eps(1e-15).betas(std::make_tuple(0.9, 0.99));
			if (fused_adam) opt = std::make_unique<FusedAdam>(gv, options);
			else opt = std::make_unique<torch::optim::Adam>(gv, options);
			global_step = 0;
		}
		std::vector<double> secs; std::vector<float> losses;
		for (int i = 0; i < n_steps; i++) {
			auto t0 = std::chrono::steady_clock::now();
			auto p = Params(n_samples, n_importance, chunk, false, true, bbox, false, noise_std[i], sp_alpha[i]);
			opt->zero_grad();
			auto r = renderer->Render(0, 0, Tensor(), p, {rays_o, rays_d, cone}, Tensor(), Tensor());
			auto loss = torch::nn::functional::huber_loss(r.Outputs.RGBMap, target.detach());
			loss.backward();
			opt->step();
			const float new_lr = lr * powf(0.1f, float(global_step) / (lrate_decay * 1000));
			for (auto& g : opt->param_groups()) g.options().set_lr(new_lr);
			global_step++;
			const float lv = loss.template item<float>();
			secs.push_back(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
			losses.push_back(lv);
		}
		return {secs, losses};
	}
	/// kernels of the training graph's last step (0 before the first graph step)
	int GraphKernels() { return graph ? graph->KernelsPerStep() : 0; }
};

// The language branch of NeRFExecutor (src/NeRFExecutor.h:458-470, 504-523, 531-535, 640-650, 957-983): second CuHashEmbedder + LeRF + LeRFRenderer
struct OpenLeRFRenderer : public LeRFRenderer {
	using LeRFRenderer::LeRFRenderer;
	using LeRFRenderer::RunLENetwork;
	using LeRFRenderer::RawToLEOutputs;
};

static py::dict ToDict(const LeRFRendererOutputs& o)
{
	py::dict d;
	d["rendered"] = o.RenderedLangEmbedding; d["embedding"] = o.LangEmbedding; d["weights"] = o.WeightsLE; d["depth"] = o.DepthMapLE;
	d["disp"] = o.DispMapLE; d["acc"] = o.AccMapLE; d["relevancy"] = o.Relevancy;
	return d;
}

struct LerfPipe {
	CuHashEmbedder embed{nullptr};
	LeRF model{nullptr};
	std::unique_ptr<OpenLeRFRenderer> renderer;
	std::unique_ptr<torch::optim::Adam> opt;
	Tensor bbox;

	void Finish()
	{
		embed->to(torch::kCUDA); model->to(torch::kCUDA);
		renderer = std::make_unique<OpenLeRFRenderer>(embed, model);
	}
	std::vector<Tensor> EmbedParams() { return embed->parameters(); }
	std::vector<Tensor> ModelParams() { return model->parameters(); }
	std::vector<std::string> ModelParamNames() { std::vector<std::string> r; for (auto& p : model->named_parameters()) r.push_back(p.key()); return r; }
	void InitModel() { Trainable::Initialize(model); }
	Tensor Model(Tensor x) { return model->forward(x); }
	Tensor RunLENetwork(Tensor pts) { return renderer->RunLENetwork(pts, model, embed); }
	py::dict RawToLEOutputs(Tensor raw_le, Tensor z, Tensor rays_d) { return ToDict(renderer->RawToLEOutputs(raw_le, z, rays_d, model->GetLangEmbedDim(), 0.f)); }
	py::dict Render(Tensor rays_o, Tensor rays_d, int n_samples, int n_importance, int chunk, bool materialize, bool return_raw)
	{
		auto p = Params(n_samples, n_importance, chunk, false, false, bbox, true, 0.f, 0.f);
		p.ReturnRaw = return_raw;
		renderer->MaterializeLangEmbedding = materialize;
		auto r = renderer->Render(0, 0, Tensor(), p, {rays_o, rays_d, Tensor()}, Tensor(), Tensor());
		py::dict d = ToDict(r.Outputs);
		d["near"] = r.Near; d["far"] = r.Far; d["raw"] = r.Raw;
		return d;
	}
	/// the language lines of NeRFExecutor::Train (src/NeRFExecutor.h:957-983, 986): Render, huber(delta 1.25).sum(-1).nanmean(), backward, Adam
	std::vector<float> TrainSteps(Tensor rays_o, Tensor rays_d, Tensor target, int n_steps, int n_samples, int n_importance, int chunk, float lr)
	{
		if (!opt) {
			std::vector<Tensor> gv;
			for (auto& p : embed->parameters()) gv.push_back(p);
			for (auto& p : model->parameters()) gv.push_back(p);
			opt = std::make_unique<torch::optim::Adam>(gv, torch::optim::AdamOptions(lr).eps(1e-15).betas(std::make_tuple(0.9, 0.99)));
		}
		std::vector<float> losses;
		auto p = Params(n_samples, n_importance, chunk, false, false, bbox, true, 0.f, 0.f);
		for (int i = 0; i < n_steps; i++) {
			opt->zero_grad();
			auto r = renderer->Render(0, 0, Tensor(), p, {rays_o, rays_d, Tensor()}, Tensor(), Tensor());
			auto loss = torch::nn::functional::huber_loss(r.Outputs.RenderedLangEmbedding, target.detach(),
				torch::nn::functional::HuberLossFuncOptions().reduction(torch::kNone).delta(1.25)).sum(-1).nanmean();
			loss.backward();
			opt->step();
			losses.push_back(loss.item<float>());
		}
		return losses;
	}
};

using CuHashPipe = Pipeline<CuHashEmbedder, CuSHEncoder, NeRFSmall>;
using ClassicPipe = Pipeline<Embedder, Embedder, NeRF>;

template <class P>
static void Bind(py::module_& m, const char* name)
{
	py::class_<P>(m, name)
		.def("embed_params", &P::EmbedParams).def("model_params", &P::ModelParams).def("model_param_names", &P::ModelParamNames)
		.def("embed_param_names", &P::EmbedParamNames).def("embed_buffers", &P::EmbedBuffers).def("embed_buffer_names", &P::EmbedBufferNames)
		.def("init_model", &P::InitModel).def("output_dims", &P::OutputDims)
		.def("embed", &P::Embed).def("embed_dirs", &P::EmbedDirs).def("model", &P::Model)
		.def("run_network", &P::RunNetwork).def("raw_to_outputs", &P::RawToOutputs)
		.def("render_rays", &P::RenderRays).def("render", &P::Render).def("render_shipped", &P::RenderShipped).def("render_image", &P::RenderImage)
		.def("use_fused_adam", &P::UseFusedAdam).def("use_train_graph", &P::UseTrainGraph)
		.def("use_fused_inference", [](P& p, bool on) { p.renderer->UseFusedInference = on; })
		.def("reuse_coarse_rows", [](P& p, bool on) { p.renderer->ReuseCoarseRows = on; })
		.def("train_steps", &P::TrainSteps, py::call_guard<py::gil_scoped_release>())
		.def("train_steps_shipped", &P::TrainStepsShipped, py::call_guard<py::gil_scoped_release>())
		.def("graph_kernels", &P::GraphKernels)
		// NeRFExecutor::SaveCheckpoint / the restore branch of Initialize (src/NeRFExecutor.h:1054-1068, 546-553): same file names
		.def("save_checkpoint", [](P& p, const std::string& dir) {
			torch::save(p.embed, dir + "/embedder_checkpoint.pt");
			torch::save(p.model, dir + "/model_checkpoint.pt");
		})
		.def("load_checkpoint", [](P& p, const std::string& dir) {
			torch::load(p.embed, dir + "/embedder_checkpoint.pt");
			torch::load(p.model, dir + "/model_checkpoint.pt");
		});
}

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m)
{
	m.doc() = "nerfpp_b200 C++ drop-in layer (torch::Tensor boundary over the sm_100a C ABI)";
	m.def("manual_seed", [](int64_t s) { torch::manual_seed(s); });
	m.def("trunc_exp", [](Tensor x) { return torch::autograd::TruncExp::apply(x)[0]; });
	m.def("sample_pdf", &SamplePDF);
	m.def("intersect_aabb", [](Tensor o, Tensor d, Tensor bbox, float near_plane) { return IntersectWithAABB(o, d, bbox, near_plane); });
	m.def("get_rays", [](int h, int w, Tensor k, Tensor c2w) { return GetRays(h, w, k, c2w); });
	m.def("embedder", [](Tensor x, int multires) { Embedder e("embedder", multires); return e->forward(x).first; });
	m.def("cu_sh_encoder", [](Tensor x, int degree) { CuSHEncoder e("embeddirs", 3, degree); return e->forward(x).first; });
	m.def("tangent_scatter", [](Tensor pts, Tensor z, Tensor cone, Tensor d, Tensor bbox) { return TangentScatter(pts, z, cone, d, pts.device(), bbox); });
	m.def("reflect_boundary", &ReflectBoundary);
	m.def("total_variation_loss", [](CuHashPipe& p) { return TotalVariationLoss(p.embed); });

	m.def("invalidate_caches", [](CuHashPipe& p) { p.embed->InvalidateCaches(); p.model->InvalidateCaches(); });
	m.def("classic_invalidate_caches", [](ClassicPipe& p) { p.model->InvalidateCaches(); });
	m.def("lerf_invalidate_caches", [](LerfPipe& p) { p.embed->InvalidateCaches(); p.model->InvalidateCaches(); });
	m.def("classic_set_fused_training", [](ClassicPipe& p, bool on) { p.model->FusedTraining = on; });
	m.def("classic_set_fused_embedding", [](ClassicPipe& p, bool on) { p.model->FusedEmbedding = on; });
	Bind<CuHashPipe>(m, "CuHashPipe");
	Bind<ClassicPipe>(m, "ClassicPipe");
	m.def("make_cuhash", [](Tensor bbox, int n_levels, int n_feat, int log2_t, int base_res, int finest_res, int sh_degree, int num_layers,
		int hidden, int geo_feat, int num_layers_color, int hidden_color) {
		auto p = std::make_unique<CuHashPipe>();
		p->bbox = bbox;
		p->embed = CuHashEmbedder("embedder", bbox, n_levels, n_feat, log2_t, base_res, finest_res);
		p->embeddirs = CuSHEncoder("embeddirs", 3, sh_degree);
		p->model = NeRFSmall(num_layers, hidden, geo_feat, num_layers_color, hidden_color, false, 3, 64, p->embed->GetOutputDims(),
			p->embeddirs->GetOutputDims(), "model");
		p->Finish();
		return p;
	});
	py::class_<LerfPipe>(m, "LerfPipe")
		.def("embed_params", &LerfPipe::EmbedParams).def("model_params", &LerfPipe::ModelParams).def("model_param_names", &LerfPipe::ModelParamNames)
		.def("init_model", &LerfPipe::InitModel).def("model", &LerfPipe::Model).def("run_le_network", &LerfPipe::RunLENetwork)
		.def("raw_to_le_outputs", &LerfPipe::RawToLEOutputs).def("render", &LerfPipe::Render)
		.def("train_steps", &LerfPipe::TrainSteps, py::call_guard<py::gil_scoped_release>())
		// A/B: false routes training through the reference's formulation (torch::linear + LibTorch autograd) instead of the fused backward
		.def("use_fused_training", [](LerfPipe& p, bool on) { p.renderer->UseFusedTraining = on; })
		.def("language_grads", [](LerfPipe& p, Tensor rays_o, Tensor rays_d, Tensor target, int n_samples, int n_importance) {
			// one backward of the language loss (src/NeRFExecutor.h:957-983) without an optimiser step: (loss, d embeddings, d weights...)
			for (auto& t : p.embed->parameters()) if (t.grad().defined()) t.mutable_grad().zero_();
			for (auto& t : p.model->parameters()) if (t.grad().defined()) t.mutable_grad().zero_();
			auto prm = Params(n_samples, n_importance, 1 << 20, false, false, p.bbox, true, 0.f, 0.f);
			auto r = p.renderer->Render(0, 0, Tensor(), prm, {rays_o, rays_d, Tensor()}, Tensor(), Tensor());
			auto loss = torch::nn::functional::huber_loss(r.Outputs.RenderedLangEmbedding, target.detach(),
				torch::nn::functional::HuberLossFuncOptions().reduction(torch::kNone).delta(1.25)).sum(-1).nanmean();
			loss.backward();
			std::vector<Tensor> g;
			for (auto& t : p.embed->parameters()) g.push_back(t.grad().clone());
			for (auto& t : p.model->parameters()) g.push_back(t.grad().clone());
			return std::make_pair(loss.item<float>(), g);
		}, py::call_guard<py::gil_scoped_release>())
		// NeRFExecutor::SaveCheckpoint / restore for the language branch (src/NeRFExecutor.h:556-560, 574-578, 1062-1066): same file names
		.def("save_checkpoint", [](LerfPipe& p, const std::string& dir) {
			torch::save(p.embed, dir + "/lang_embedder_checkpoint.pt");
			torch::save(p.model, dir + "/lang_model_checkpoint.pt");
		})
		.def("load_checkpoint", [](LerfPipe& p, const std::string& dir) {
			torch::load(p.embed, dir + "/lang_embedder_checkpoint.pt");
			torch::load(p.model, dir + "/lang_model_checkpoint.pt");
		});
	// src/NeRFExecutor.h:461 and :507-514
	m.def("make_lerf", [](Tensor bbox, int n_levels, int n_feat, int log2_t, int base_res, int finest_res, int geo_feat, int num_layers, int hidden,
		int lang_dim) {
		auto p = std::make_unique<LerfPipe>();
		p->bbox = bbox;
		p->embed = CuHashEmbedder("lang_embedder", bbox, n_levels, n_feat, log2_t, base_res, finest_res);
		p->model = LeRF(geo_feat, num_layers, hidden, lang_dim, p->embed->GetOutputDims(), "lang_model");
		p->Finish();
		return p;
	});
	m.def("make_classic", [](Tensor bbox, int multires, int multires_views, int depth, int width, bool use_viewdirs) {
		auto p = std::make_unique<ClassicPipe>();
		p->bbox = bbox;
		p->embed = Embedder("embedder", multires);
		p->embeddirs = Embedder("embeddirs", multires_views);
		p->model = NeRF(depth, width, p->embed->GetOutputDims(), p->embeddirs->GetOutputDims(), 5, std::set<int>{4}, use_viewdirs, "model");
		p->Finish();
		return p;
	});
}
