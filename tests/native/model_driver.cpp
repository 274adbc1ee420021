// tests/native/model_driver.cpp -- TEST INFRASTRUCTURE ONLY.
// Drives the UNMODIFIED reference Model (model.cpp compiled from the reference tree).  Built twice:
//  (1) oracle/Makefile -> oracle/_ref/libopensplat_ref_model.so: model.cpp + the reference's own CPU operators; pins the
//      restatements in oracle/scene_edit.py against the reference itself (torch.ops.opensplat_ref_model.*);
//  (2) oracle/build_model_b200.py -> oracle/_ref/libopensplat_model_b200.so: the SAME unmodified model.cpp compiled
//      with -DUSE_CUDA against THIS repo's operator layer (csrc/ops) -- the drop-in check that Model::forward /
//      mainLoss / optimizersStep / afterTrain run unchanged on the B200 back end (torch.ops.opensplat_b200_model.*).
//   after_train   -> Model::afterTrain  (model.cpp:311-500), incl. the Adam-state surgery
//   save          -> Model::save        (model.cpp:496-594; .ply or .splat by extension)
//   train         -> the body of the reference's training loop (opensplat.cpp:151-170) for a few steps
//   load          -> Model::loadPly     (model.cpp:614-778)
//   train_fused   -> (build (2) only) the same loop with the opt-in one-liners of csrc/ops/fused_extras.hpp in place of
//                    the bodies of Model::forward and Model::mainLoss; everything else (optimizers, schedulers,
//                    afterTrain) is still the reference's code
// Nothing of the reference is copied: a Model is constructed through its own constructor (with a stub for the
// nanoflann-based PointsTensor::scales(), whose result we overwrite anyway), its public tensors are replaced by the
// caller's, its optimizers are re-created by its own setupOptimizers(), and the Adam moments are injected as the
// AdamParamState entries that Model::addToOptimizer / removeFromOptimizer read.
#include <torch/torch.h>
#include <torch/library.h>

#include "model.hpp"
#ifdef GSB_DRIVER_FUSED
#include "fused_extras.hpp"   // the opt-in fused operators of the B200 operator layer (csrc/ops)
#endif

// ---- symbols of reference translation units we do not link (never reached by the calls above) ----
torch::Tensor PointsTensor::scales() { return torch::ones({tensor.size(0), 1}, torch::kFloat32); }
PointsTensor::~PointsTensor() {}

namespace {

using torch::Tensor;

void inject_state(torch::optim::Adam *opt, const Tensor &m, const Tensor &v) {
    Tensor param = opt->param_groups()[0].params()[0];
    auto st = std::make_unique<torch::optim::AdamParamState>();
    st->step(1);
    st->exp_avg(m.clone());
    st->exp_avg_sq(v.clone());
    opt->state()[param.unsafeGetTensorImpl()] = std::move(st);
}

std::pair<Tensor, Tensor> read_state(torch::optim::Adam *opt) {
    Tensor param = opt->param_groups()[0].params()[0];
    auto &st = static_cast<torch::optim::AdamParamState &>(*opt->state()[param.unsafeGetTensorImpl()]);
    return {st.exp_avg().clone(), st.exp_avg_sq().clone()};
}

std::unique_ptr<Model> make_model(const std::vector<Tensor> &params, int64_t numCameras, int64_t refineEvery,
                                  int64_t warmupLength, int64_t resetAlphaEvery, double densifyGradThresh,
                                  double densifySizeThresh, int64_t stopScreenSizeAt, double splitScreenSize,
                                  int64_t maxSteps, bool keepCrs, double scale, const Tensor &translation,
                                  int64_t shDegreeInterval = 1000) {
    const int64_t n = params[0].size(0);
    const int64_t restBases = params[4].size(1);
    int shDegree = 0;
    while ((shDegree + 1) * (shDegree + 1) < restBases + 1) ++shDegree;
    InputData in;
    in.scale = (float)scale;
    in.translation = translation.clone();
    in.points.xyz = torch::zeros({n, 3}, torch::kFloat32);
    in.points.rgb = torch::zeros({n, 3}, torch::kUInt8);
    const torch::Device device = params[0].device();
    auto m = std::make_unique<Model>(in, (int)numCameras, /*numDownscales*/ 0, /*resolutionSchedule*/ 3000, shDegree,
                                     (int)shDegreeInterval, (int)refineEvery, (int)warmupLength,
                                     (int)resetAlphaEvery, (float)densifyGradThresh, (float)densifySizeThresh,
                                     (int)stopScreenSizeAt, (float)splitScreenSize, (int)maxSteps, keepCrs, device);
    m->means = params[0].detach().clone().requires_grad_();
    m->scales = params[1].detach().clone().requires_grad_();
    m->quats = params[2].detach().clone().requires_grad_();
    m->featuresDc = params[3].detach().clone().requires_grad_();
    m->featuresRest = params[4].detach().clone().requires_grad_();
    m->opacities = params[5].detach().clone().requires_grad_();
    m->releaseOptimizers();
    m->setupOptimizers();
    return m;
}

// params = {means, scales, quats, featuresDc, featuresRest, opacities}; adam_m / adam_v in the same order;
// stats = {} (first step after a clear) or {xysGradNorm, visCounts, max2DSize}.
// Returns params(6) + adam_m(6) + adam_v(6) + stats(3, empty tensors when cleared) after Model::afterTrain(step).
std::vector<Tensor> after_train(std::vector<Tensor> params, std::vector<Tensor> adam_m, std::vector<Tensor> adam_v,
                                std::vector<Tensor> stats, Tensor xys_grad, Tensor radii, int64_t height,
                                int64_t width, int64_t step, int64_t seed, int64_t numCameras, int64_t refineEvery,
                                int64_t warmupLength, int64_t resetAlphaEvery, double densifyGradThresh,
                                double densifySizeThresh, int64_t stopScreenSizeAt, double splitScreenSize,
                                int64_t maxSteps) {
    auto m = make_model(params, numCameras, refineEvery, warmupLength, resetAlphaEvery, densifyGradThresh,
                        densifySizeThresh, stopScreenSizeAt, splitScreenSize, maxSteps, false, 1.0,
                        torch::zeros({3}, torch::kFloat32));
    torch::optim::Adam *opts[6] = {m->meansOpt, m->scalesOpt, m->quatsOpt, m->featuresDcOpt, m->featuresRestOpt,
                                   m->opacitiesOpt};
    for (int i = 0; i < 6; ++i) inject_state(opts[i], adam_m[i], adam_v[i]);
    m->xys = torch::zeros_like(xys_grad).requires_grad_();
    m->xys.mutable_grad() = xys_grad.clone();
    m->radii = radii.clone();
    m->lastHeight = (int)height;
    m->lastWidth = (int)width;
    if (stats.size() == 3) {
        m->xysGradNorm = stats[0].clone();
        m->visCounts = stats[1].clone();
        m->max2DSize = stats[2].clone();
    }
    torch::manual_seed((uint64_t)seed);   // the stream Model::afterTrain's torch::randn (model.cpp:359) draws from
    m->afterTrain((int)step);
    std::vector<Tensor> out = {m->means.detach().clone(),      m->scales.detach().clone(),
                               m->quats.detach().clone(),      m->featuresDc.detach().clone(),
                               m->featuresRest.detach().clone(), m->opacities.detach().clone()};
    torch::optim::Adam *opts2[6] = {m->meansOpt, m->scalesOpt, m->quatsOpt, m->featuresDcOpt, m->featuresRestOpt,
                                    m->opacitiesOpt};
    std::vector<Tensor> ms, vs;
    for (int i = 0; i < 6; ++i) {
        auto mv = read_state(opts2[i]);
        ms.push_back(mv.first);
        vs.push_back(mv.second);
    }
    out.insert(out.end(), ms.begin(), ms.end());
    out.insert(out.end(), vs.begin(), vs.end());
    auto or_empty = [](const Tensor &t) { return t.defined() ? t.clone() : torch::empty({0}); };
    out.push_back(or_empty(m->xysGradNorm));
    out.push_back(or_empty(m->visCounts));
    out.push_back(or_empty(m->max2DSize));
    return out;
}

void save(std::vector<Tensor> params, std::string filename, int64_t step, bool keepCrs, double scale,
          Tensor translation) {
    auto m = make_model(params, 1, 100, 500, 30, 0.0002, 0.01, 4000, 0.05, 30000, keepCrs, scale, translation);
    m->save(filename, (int)step);
}

// The body of the reference's training loop (opensplat.cpp:151-170) for steps first_step .. first_step+num_steps-1,
// cameras taken round-robin: zero_grad -> Model::forward -> Model::mainLoss -> backward -> optimizersStep ->
// schedulersStep -> afterTrain.  Returns {losses [S], gaussian counts [S], last rendered image, params(6)}.
std::vector<Tensor> train_impl(bool fused, std::vector<Tensor> params, Tensor camToWorlds, Tensor gts, double fx,
                               double fy, double cx, double cy, int64_t height, int64_t width, int64_t first_step,
                               int64_t num_steps, double ssimWeight, int64_t seed, int64_t shDegreeInterval,
                               int64_t numCameras, int64_t refineEvery, int64_t warmupLength, int64_t resetAlphaEvery,
                               double densifyGradThresh, double densifySizeThresh, int64_t stopScreenSizeAt,
                               double splitScreenSize, int64_t maxSteps) {
    auto m = make_model(params, numCameras, refineEvery, warmupLength, resetAlphaEvery, densifyGradThresh,
                        densifySizeThresh, stopScreenSizeAt, splitScreenSize, maxSteps, false, 1.0,
                        torch::zeros({3}, torch::kFloat32), shDegreeInterval);
    const torch::Device device = params[0].device();
    const int64_t V = camToWorlds.size(0);
    std::vector<Camera> cams;
    for (int64_t v = 0; v < V; ++v)
        cams.emplace_back((int)width, (int)height, (float)fx, (float)fy, (float)cx, (float)cy, 0.f, 0.f, 0.f, 0.f, 0.f,
                          camToWorlds[v].to(torch::kCPU).clone(), "");
    torch::manual_seed((uint64_t)seed);
    std::vector<float> losses;
    std::vector<int64_t> counts;
    Tensor rgb;
    for (int64_t step = first_step; step < first_step + num_steps; ++step) {
        const int64_t v = (step - 1) % V;
        m->optimizersZeroGrad();
        Tensor gt = gts[v].to(device);
        Tensor loss;
#ifdef GSB_DRIVER_FUSED
        if (fused) {
            // what the bodies of Model::forward / Model::mainLoss become when a maintainer opts in (INTEGRATION.md)
            Camera &cam = cams[v];
            const float sf = (float)m->getDownscaleFactor((int)step);
            const int h = static_cast<int>(static_cast<float>(cam.height) / sf);
            const int w = static_cast<int>(static_cast<float>(cam.width) / sf);
            auto r = gsb::modelForward(m->means, m->scales, m->quats, m->featuresDc, m->featuresRest, m->opacities,
                                       m->backgroundColor, cam.camToWorld, cam.fx / sf, cam.fy / sf, cam.cx / sf,
                                       cam.cy / sf, h, w, (std::min<int>)((int)step / m->shDegreeInterval, m->shDegree));
            m->xys = r.xys;
            m->radii = r.radii;
            m->lastHeight = h;
            m->lastWidth = w;
            rgb = r.rgb;
            loss = gsb::MainLoss::apply(rgb, gt, ssimWeight);
        } else
#endif
        {
            rgb = m->forward(cams[v], (int)step);
            loss = m->mainLoss(rgb, gt, (float)ssimWeight);
        }
        loss.backward();
        losses.push_back(loss.item<float>());
        m->optimizersStep();
        m->schedulersStep((int)step);
        m->afterTrain((int)step);
        counts.push_back(m->means.size(0));
    }
    std::vector<Tensor> out = {torch::tensor(losses), torch::tensor(counts), rgb.detach().clone(),
                               m->means.detach().clone(),      m->scales.detach().clone(),
                               m->quats.detach().clone(),      m->featuresDc.detach().clone(),
                               m->featuresRest.detach().clone(), m->opacities.detach().clone()};
    return out;
}

std::vector<Tensor> train(std::vector<Tensor> params, Tensor camToWorlds, Tensor gts, double fx, double fy, double cx,
                          double cy, int64_t height, int64_t width, int64_t first_step, int64_t num_steps,
                          double ssimWeight, int64_t seed, int64_t shDegreeInterval, int64_t numCameras,
                          int64_t refineEvery, int64_t warmupLength, int64_t resetAlphaEvery, double densifyGradThresh,
                          double densifySizeThresh, int64_t stopScreenSizeAt, double splitScreenSize, int64_t maxSteps) {
    return train_impl(false, params, camToWorlds, gts, fx, fy, cx, cy, height, width, first_step, num_steps, ssimWeight,
                      seed, shDegreeInterval, numCameras, refineEvery, warmupLength, resetAlphaEvery, densifyGradThresh,
                      densifySizeThresh, stopScreenSizeAt, splitScreenSize, maxSteps);
}

#ifdef GSB_DRIVER_FUSED
std::vector<Tensor> train_fused(std::vector<Tensor> params, Tensor camToWorlds, Tensor gts, double fx, double fy,
                                double cx, double cy, int64_t height, int64_t width, int64_t first_step,
                                int64_t num_steps, double ssimWeight, int64_t seed, int64_t shDegreeInterval,
                                int64_t numCameras, int64_t refineEvery, int64_t warmupLength, int64_t resetAlphaEvery,
                                double densifyGradThresh, double densifySizeThresh, int64_t stopScreenSizeAt,
                                double splitScreenSize, int64_t maxSteps) {
    return train_impl(true, params, camToWorlds, gts, fx, fy, cx, cy, height, width, first_step, num_steps, ssimWeight,
                      seed, shDegreeInterval, numCameras, refineEvery, warmupLength, resetAlphaEvery, densifyGradThresh,
                      densifySizeThresh, stopScreenSizeAt, splitScreenSize, maxSteps);
}
#endif

// Model::loadPly (model.cpp:614-778) -> {step (int64 scalar), means, scales, quats, featuresDc, featuresRest, opacities}
std::vector<Tensor> load(std::string filename, bool keepCrs, double scale, Tensor translation, Tensor like) {
    std::vector<Tensor> dummy = {torch::zeros({1, 3}, like.options()), torch::zeros({1, 3}, like.options()),
                                 torch::ones({1, 4}, like.options()),  torch::zeros({1, 3}, like.options()),
                                 torch::zeros({1, 15, 3}, like.options()), torch::zeros({1, 1}, like.options())};
    auto m = make_model(dummy, 1, 100, 500, 30, 0.0002, 0.01, 4000, 0.05, 30000, keepCrs, scale, translation);
    const int step = m->loadPly(filename);
    return {torch::tensor((int64_t)step),      m->means.detach().clone(),        m->scales.detach().clone(),
            m->quats.detach().clone(),         m->featuresDc.detach().clone(),   m->featuresRest.detach().clone(),
            m->opacities.detach().clone()};
}

}  // namespace

#ifndef GSB_DRIVER_LIB
#define GSB_DRIVER_LIB opensplat_ref_model
#endif

TORCH_LIBRARY(GSB_DRIVER_LIB, m) {
    m.def("after_train", &after_train);
    m.def("save", &save);
    m.def("train", &train);
#ifdef GSB_DRIVER_FUSED
    m.def("train_fused", &train_fused);
#endif
    m.def("load", &load);
}
