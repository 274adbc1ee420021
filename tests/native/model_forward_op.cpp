// tests/native/model_forward_op.cpp -- TEST INFRASTRUCTURE ONLY.
// Exposes gsb::modelForward (csrc/ops/fused_extras.hpp), the opt-in body of Model::forward, to Python as
// torch.ops.opensplat_b200_test.model_forward, so that tests/test_gpu_model.py can drive it -- camera matrices formed on
// the host, tile bounds, the background early return and all -- inside a training loop.  Built from this repo's sources
// only (opensplat_b200/build_ops.py build_test_ops -> tests/native/_build/libopensplat_b200_test_ops.so).
#include <torch/library.h>

#include "fused_extras.hpp"

namespace {

// -> {rgb [H, W, 3], xys [N, 2] (retain_grad set), radii [N]}
std::vector<torch::Tensor> model_forward(torch::Tensor means, torch::Tensor logScales, torch::Tensor rawQuats,
                                         torch::Tensor featuresDc, torch::Tensor featuresRest,
                                         torch::Tensor opacityLogits, torch::Tensor backgroundColor,
                                         torch::Tensor camToWorld, double fx, double fy, double cx, double cy,
                                         int64_t height, int64_t width, int64_t degreesToUse) {
    auto r = gsb::modelForward(means, logScales, rawQuats, featuresDc, featuresRest, opacityLogits, backgroundColor,
                               camToWorld, (float)fx, (float)fy, (float)cx, (float)cy, (int)height, (int)width,
                               (int)degreesToUse);
    return {r.rgb, r.xys, r.radii};
}

}  // namespace

TORCH_LIBRARY(opensplat_b200_test, m) { m.def("model_forward", &model_forward); }
