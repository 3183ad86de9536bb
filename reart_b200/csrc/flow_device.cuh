// flow_device.cuh -- the per-component rule of the flow loss (run_robot.py:194-213, networks/loss.py:10-21), shared by
// kin_flow_kernel (kin.cu: the gradient summed per (frame, part) of the kinematic model) and flow_grad_kernel (flow.cu: the
// gradient per point of the skinned cloud), so both kernels compute every term with the same operations.
#pragma once
#include <cuda_runtime.h>

namespace reart {

constexpr float kFlowSmoothWeight = 1e-2f;                   // networks/loss.py:10 smooth_weight

// d flow_loss / d pred (one component) and the per-component loss term
__device__ __forceinline__ float flow_term_grad(float pred, float tgt, bool keep, int robust, float& term) {
    if (!keep) {
        term = kFlowSmoothWeight * (pred * pred);
        return 2.0f * kFlowSmoothWeight * pred;
    }
    const float e = pred - tgt;
    if (!robust) {
        term = e * e;
        return 2.0f * e;
    }
    const float a = fabsf(e);
    if (a < 1.0f) {                                           // torch.where(a < 1, ...): |err| == 1 is the linear branch
        term = 0.5f * e * e;
        return e;
    }
    term = a - 0.5f;
    return e > 0.f ? 1.0f : -1.0f;
}

}  // namespace reart
