// flow.cu -- the flow loss of run_robot.py:194-213 (networks/loss.py:10-21) and its gradient w.r.t. the skinned cloud, on a
// window of K consecutive frames of the complete sequence, for a model whose weights train (the relaxation model: the
// gradient goes on through reart_skin_bwd to gW, gR, gtr).  Slot s holding local frame t, point i, component r:
//   pred_k = win[k+1] - win[k],  d_k = d flow_loss / d pred_k (flow_term_grad, shared with kin_flow_kernel)
//   g_skinned[t,i,r] (+)= lambda (d_{s-1} - d_s)   (a pair outside the window is dropped)
// kin_flow_kernel's formula without the sum over the part's points.  A CTA per (slot, chunk of 256 points), one point per
// thread: the gradient needs no sum at all.  Pair k's loss is counted (if q0 <= k < q1) by slot k+1 when that slot is
// local, else by slot k, as kin_flow_kernel counts it.  The loss: a fixed xor tree per warp, the warps in order, per-CTA
// double partials added in index order by the last CTA (ticket, re-armed for graph replay).  No float atomics.
#include "common.cuh"
#include "flow_device.cuh"
#include "kernels.h"

namespace reart {

constexpr int kFlowGradThreads = 256;

int64_t flow_grad_blocks(int64_t K, int64_t N) { return K * ceil_div(N, (int64_t)kFlowGradThreads); }

__global__ void __launch_bounds__(kFlowGradThreads) flow_grad_kernel(const FlowGrad a) {
    constexpr int kWarps = kFlowGradThreads / 32;
    __shared__ double s_loss[kWarps];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int s = blockIdx.y, K = a.K;
    const int64_t N = a.N;
    const int64_t i = (int64_t)blockIdx.x * kFlowGradThreads + threadIdx.x;
    const int t = a.slot_frame[s];
    double loss = 0.0;
    if (t >= 0 && t < a.T && i < N) {
        const bool has_prev = s > 0, has_next = s < K - 1;
        const bool count_prev = has_prev && s - 1 >= a.q0 && s - 1 < a.q1;           // slot s is the pair's second slot
        const bool count_next = has_next && s >= a.q0 && s < a.q1 && a.slot_frame[s + 1] < 0;
        const float* ws = a.win + ((int64_t)s * N + i) * 3;
        float g[3] = {0.f, 0.f, 0.f};
        float lp = 0.f, ln = 0.f;
        if (has_prev) {
            const float* wp = ws - N * 3;
            const float* tf = a.tflow + ((int64_t)(s - 1) * N + i) * 3;
            const bool keep = a.mask[(int64_t)(s - 1) * N + i] != 0;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                float term;
                g[r] = flow_term_grad(ws[r] - wp[r], tf[r], keep, a.robust, term);
                lp += term;
            }
        }
        if (has_next) {
            const float* wn = ws + N * 3;
            const float* tf = a.tflow + ((int64_t)s * N + i) * 3;
            const bool keep = a.mask[(int64_t)s * N + i] != 0;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                float term;
                g[r] -= flow_term_grad(wn[r] - ws[r], tf[r], keep, a.robust, term);
                ln += term;
            }
        }
        if (count_prev) loss += (double)lp;
        if (count_next) loss += (double)ln;
        float* o = a.g_skinned + ((int64_t)t * N + i) * 3;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float v = __fmul_rn(a.lambda, g[r]);         // not contracted: accumulate is exactly one float add
            o[r] = a.accumulate ? o[r] + v : v;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, o);
    if (lane == 0) s_loss[w] = loss;
    __syncthreads();
    const int nblk = gridDim.x * gridDim.y, blk = blockIdx.y * gridDim.x + blockIdx.x;
    if (threadIdx.x == 0) {
        double c = 0.0;
#pragma unroll
        for (int q = 0; q < kWarps; ++q) c += s_loss[q];
        a.partials[blk] = c;
        __threadfence();
        s_last = atomicAdd(a.ticket, 1u) == (unsigned)nblk - 1u;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        const volatile double* v = a.partials;
        double tot = 0.0;
        for (int b = 0; b < nblk; ++b) tot += v[b];
        *a.loss = a.accumulate ? *a.loss + (double)a.lambda * tot : (double)a.lambda * tot;
        *a.ticket = 0u;                                       // re-armed for the next launch (graph replay)
    }
}

int launch_flow_grad(const FlowGrad& a, cudaStream_t stream) {
    if (a.T <= 0) return kOk;
    if (a.K < 2 || a.N <= 0) return kErrInvalidArg;
    dim3 grid((unsigned)ceil_div(a.N, kFlowGradThreads), (unsigned)a.K);
    flow_grad_kernel<<<grid, kFlowGradThreads, 0, stream>>>(a);
    REART_CHECK_LAUNCH();
    return kOk;
}

}  // namespace reart
