// kin.cu -- one iteration of the kinematic (projection) model, run_robot.py's second model (--model=kinematic,
// networks/model.py:73-166), around the fused energy of capi.cu:
//
//   head = tree forward kinematics (utils/kinematic_utils.py:151-198) + the optional learned root pose
//          (networks/model.py:151-159): R [T,P,3,3], tr [T,P,3] for the energy, the per-part poses before the root pose
//          for the backward.  The arithmetic is fk_fwd_kernel's (screw_eval<float>, mat34_mul), so without a root pose
//          R / tr are bit-identical to reart_fk_fwd.
//   tail = root-pose backward + FK backward (the dual-number screw of fk_bwd_kernel) + the frame sums of the shared
//          gradients in frame order + [the one-shot all-reduce of allreduce.cu, inline, when frames are sharded]
//          + Adam (torch.optim.Adam semantics, one parameter group) on every parameter.
// The work is T*P small dependent steps: the tail is ONE CTA striding over frames.  No float atomics anywhere, so a step
// is bit-reproducible (fk_bwd_kernel's atomicAdd over frames is what the autograd path does instead).
#include "common.cuh"
#include "flow_device.cuh"
#include "kernels.h"
#include "se3_device.cuh"
#include "tail_device.cuh"

namespace reart {

// ============================================================================================ head
constexpr int kKinHeadThreads = 32;                          // one thread per frame, as fk_fwd_kernel

__global__ void __launch_bounds__(kKinHeadThreads) kin_head_kernel(const FkParams p, const float* __restrict__ root_6d,
                                                                   const float* __restrict__ root_t, float* __restrict__ R,
                                                                   float* __restrict__ tr, float* __restrict__ fk) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.T) return;
    const bool has_root = root_6d != nullptr;
    float root[12];                                           // [R_root | t_root], 3x4
    if (has_root) {
        float in[6], Rr[9];
#pragma unroll
        for (int k = 0; k < 6; ++k) in[k] = root_6d[(int64_t)t * 6 + k];
        rot6d_eval<float>(in, Rr);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            root[4 * i] = Rr[3 * i]; root[4 * i + 1] = Rr[3 * i + 1]; root[4 * i + 2] = Rr[3 * i + 2];
            root[4 * i + 3] = root_t[(int64_t)t * 3 + i];
        }
    }
    for (int oi = 0; oi < p.P; ++oi) {
        const int c = p.order[oi];
        const int par = p.parent[c];
        float M[12];
        if (par < 0) {
            for (int k = 0; k < 12; ++k) M[k] = (k % 5 == 0) ? 1.f : 0.f;
        } else {
            const int e = p.edge[c];
            float th, dd; bool tv, dv;
            fk_joint_inputs(p, t, e, th, dd, tv, dv);
            float L[3] = {p.axis[3 * e], p.axis[3 * e + 1], p.axis[3 * e + 2]};
            float Mo[3] = {p.moment[3 * e], p.moment[3 * e + 1], p.moment[3 * e + 2]};
            float rel[12];
            screw_eval<float>(L, Mo, th, dd, rel);
            mat34_mul(fk + ((int64_t)t * p.P + par) * 12, rel, M);
        }
        float* F = fk + ((int64_t)t * p.P + c) * 12;
        for (int k = 0; k < 12; ++k) F[k] = M[k];
        float out[12];
        if (has_root) mat34_mul(root, M, out);                // networks/model.py:157-158: root @ fk
        else for (int k = 0; k < 12; ++k) out[k] = M[k];
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) R[((int64_t)t * p.P + c) * 9 + 3 * i + j] = out[4 * i + j];
            tr[((int64_t)t * p.P + c) * 3 + i] = out[4 * i + 3];
        }
    }
}

int launch_kin_head(const FkParams& p, const float* root_6d, const float* root_t, float* R, float* tr, float* fk,
                    cudaStream_t stream) {
    if (p.T <= 0) return kOk;
    if (p.P <= 0 || p.P > 32) return kErrUnsupported;
    kin_head_kernel<<<(unsigned)ceil_div(p.T, kKinHeadThreads), kKinHeadThreads, 0, stream>>>(p, root_6d, root_t, R, tr, fk);
    REART_CHECK_LAUNCH();
    return kOk;
}

// ============================================================================================ tail
constexpr int kKinTailThreads = 256;

int64_t kin_tail_workspace_floats(int64_t T, int64_t P) { return T * 6 * (P - 1) + T * P * 12; }

__global__ void __launch_bounds__(kKinTailThreads) kin_tail_kernel(const KinTail a) {
    __shared__ int s_ok;
    const int T = a.T, P = a.P, E = P - 1;
    const int nshared = 6 * E;                                // [g_axis | g_moment], then the loss
    const int o_theta = nshared + 1;
    const int o_dist = o_theta + T * E;
    const int o_d6 = o_dist + (a.distance ? T * E : 0);
    const int o_rt = o_d6 + 6 * T;
    const int n_grad = o_d6 + (a.root_6d ? 9 * T : 0);
    float* g = a.grad;
    float* fpart = a.partials;                                // [T][6E] per-frame shared-gradient terms
    float* work = a.partials + (int64_t)T * nshared;          // [T][P][12] dL/d (pose before the root pose)
    if (a.phase != 2) {
        const FkParams fp = {a.axis, a.moment, a.theta, a.distance, a.order, a.parent, a.edge, a.joint_type, T, P};
        for (int t = threadIdx.x; t < T; t += blockDim.x) {
            float* gw = work + (int64_t)t * P * 12;
            const float* gR = a.gR + (int64_t)t * P * 9;
            const float* gT = a.gtr + (int64_t)t * P * 3;
            if (a.root_6d) {
                // out_c = [Rr | tr] [F_c; 0001]:  dL/dF_c = Rr^T G_c,  dL/dRr = sum_c G_c F_c^T (3x4 . 4x3),  dL/dtr = sum_c G_c[:,3]
                Dual<6> in[6], Rr[9];
#pragma unroll
                for (int k = 0; k < 6; ++k) in[k] = Dual<6>::var(a.root_6d[(int64_t)t * 6 + k], k);
                rot6d_eval<Dual<6>>(in, Rr);
                float gRr[9], gtr[3] = {0.f, 0.f, 0.f};
#pragma unroll
                for (int k = 0; k < 9; ++k) gRr[k] = 0.f;
                for (int c = 0; c < P; ++c) {
                    const float* F = a.fk + ((int64_t)t * P + c) * 12;
                    float G[12];
#pragma unroll
                    for (int i = 0; i < 3; ++i) {
                        G[4 * i] = gR[c * 9 + 3 * i]; G[4 * i + 1] = gR[c * 9 + 3 * i + 1]; G[4 * i + 2] = gR[c * 9 + 3 * i + 2];
                        G[4 * i + 3] = gT[c * 3 + i];
                    }
#pragma unroll
                    for (int i = 0; i < 3; ++i) {
#pragma unroll
                        for (int k = 0; k < 3; ++k)
                            gRr[3 * i + k] += G[4 * i] * F[4 * k] + G[4 * i + 1] * F[4 * k + 1] + G[4 * i + 2] * F[4 * k + 2] +
                                              G[4 * i + 3] * F[4 * k + 3];
                        gtr[i] += G[4 * i + 3];
                    }
#pragma unroll
                    for (int k = 0; k < 3; ++k)
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            gw[c * 12 + 4 * k + j] = Rr[k].v * G[j] + Rr[3 + k].v * G[4 + j] + Rr[6 + k].v * G[8 + j];
                }
                float g6[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int o = 0; o < 9; ++o)
#pragma unroll
                    for (int k = 0; k < 6; ++k) g6[k] += gRr[o] * Rr[o].d[k];
#pragma unroll
                for (int k = 0; k < 6; ++k) g[o_d6 + t * 6 + k] = g6[k];
#pragma unroll
                for (int i = 0; i < 3; ++i) g[o_rt + t * 3 + i] = gtr[i];
            } else {
                for (int c = 0; c < P; ++c)
#pragma unroll
                    for (int i = 0; i < 3; ++i) {
                        gw[c * 12 + 4 * i] = gR[c * 9 + 3 * i]; gw[c * 12 + 4 * i + 1] = gR[c * 9 + 3 * i + 1];
                        gw[c * 12 + 4 * i + 2] = gR[c * 9 + 3 * i + 2]; gw[c * 12 + 4 * i + 3] = gT[c * 3 + i];
                    }
            }
            // the tree walk of fk_bwd_kernel, leaves first; the shared terms go to this frame's row instead of atomics
            for (int oi = P - 1; oi >= 0; --oi) {
                const int c = a.order[oi];
                const int par = a.parent[c];
                if (par < 0) continue;
                const int e = a.edge[c];
                float th, dd; bool tv, dv;
                fk_joint_inputs(fp, t, e, th, dd, tv, dv);
                Dual<8> L[3], Mo[3], rel[12];
                for (int k = 0; k < 3; ++k) { L[k] = Dual<8>::var(a.axis[3 * e + k], k); Mo[k] = Dual<8>::var(a.moment[3 * e + k], 3 + k); }
                screw_eval<Dual<8>>(L, Mo, Dual<8>::var(th, 6), Dual<8>::var(dd, 7), rel);
                const float* A = a.fk + ((int64_t)t * P + par) * 12;   // parent pose
                const float* G = gw + c * 12;                         // dL/d fk[c] (complete: children were folded already)
                float* Gp = gw + par * 12;
                float g8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                for (int i = 0; i < 3; ++i) {
                    for (int j = 0; j < 4; ++j) {
                        const float dT = A[i] * G[j] + A[4 + i] * G[4 + j] + A[8 + i] * G[8 + j];
                        for (int k = 0; k < 8; ++k) g8[k] += dT * rel[4 * i + j].d[k];
                    }
                }
                for (int i = 0; i < 3; ++i) {
                    for (int j = 0; j < 4; ++j) {
                        float s = 0.f;
                        if (j < 3) s = G[4 * i] * rel[4 * j].v + G[4 * i + 1] * rel[4 * j + 1].v + G[4 * i + 2] * rel[4 * j + 2].v +
                                       G[4 * i + 3] * rel[4 * j + 3].v;
                        else s = G[4 * i + 3];
                        Gp[4 * i + j] += s;
                    }
                }
                float* row = fpart + (int64_t)t * nshared;
                for (int k = 0; k < 3; ++k) { row[3 * e + k] = g8[k]; row[3 * E + 3 * e + k] = g8[3 + k]; }
                g[o_theta + t * E + e] = tv ? g8[6] : 0.f;
                if (a.distance) g[o_dist + t * E + e] = dv ? g8[7] : 0.f;
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < nshared; i += blockDim.x) {   // sum over frames in frame order
            float s = 0.f;
            for (int t = 0; t < T; ++t) s += fpart[(int64_t)t * nshared + i];
            g[i] = s;
        }
        if (threadIdx.x == 0) g[nshared] = (float)*a.loss_local;
        __syncthreads();
    }
    if (a.phase == 1) return;                                 // the caller all-reduces g[0 .. 6E] (NCCL), then phase 2
    if (a.phase == 0 && a.world > 1)
        cta_allreduce_oneshot(a.peer_base, a.rank, a.world, nshared + 1, a.n_pad, a.epoch, g, &s_ok);
    const float step = *a.step + 1.0f;                        // 1-based index of this optimisation step
    const AdamCoef c = adam_coef(a.lr, a.beta1, a.beta2, a.eps, a.wd, step);
    for (int i = threadIdx.x; i < n_grad; i += blockDim.x) {
        if (i == nshared) continue;                           // the loss slot
        float* prm = i < 3 * E ? a.axis + i
                   : i < nshared ? a.moment + (i - 3 * E)
                   : i < o_dist ? a.theta + (i - o_theta)
                   : i < o_d6 ? a.distance + (i - o_dist)
                   : i < o_rt ? a.root_6d + (i - o_d6)
                   : a.root_t + (i - o_rt);
        adam_update(prm, a.m + i, a.v + i, g[i], c);
    }
    __syncthreads();                                          // every thread has read *a.step
    if (threadIdx.x == 0) {
        *a.loss_out = g[nshared];
        *a.step = step;
    }
}

int launch_kin_tail(const KinTail& a, cudaStream_t stream) {
    if (a.T <= 0 || a.P <= 0) return kErrInvalidArg;
    if (a.P > 32) return kErrUnsupported;
    if (a.world > 1 && a.phase == 0 && (a.world > kKinTailThreads || !a.peer_base || !a.epoch)) return kErrInvalidArg;
    kin_tail_kernel<<<1, kKinTailThreads, 0, stream>>>(a);
    REART_CHECK_LAUNCH();
    return kOk;
}

// ============================================================================================ assignment loss
// The matched-pair loss of run_robot.py:181-187 and its gradient w.r.t. the poses.  The kinematic model's skinning
// weights are one-hot rows (the label transfer), so d loss / d (R, tr) of part p in frame t is a plain sum over the
// samples of that part -- reading only the T*n sampled points instead of a [T,N,3] gradient through the full skin backward:
//   d = skinned[t, src_idx[i]] - tgt[t, col4row[t,i]],  x = cano[src_idx[i]],  g = 2 lambda d
//   loss += lambda sum |d|^2 ;  gR[t,p] += sum g x^T ;  gtr[t,p] += sum g.
// One warp per (frame, part): lane l takes the part's samples l, l+32, ... (sample_order groups them by part), then a
// fixed xor tree.  The loss: per-CTA partials, the last CTA (ticket) adds them in index order and re-arms the ticket.
constexpr int kKinAssignWarps = 4;

int64_t kin_assign_blocks(int64_t T, int64_t P) { return T * ceil_div(P, (int64_t)kKinAssignWarps); }

__global__ void __launch_bounds__(32 * kKinAssignWarps) kin_assign_kernel(const KinAssign a) {
    __shared__ double s_loss[kKinAssignWarps];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int t = blockIdx.x, p = blockIdx.y * kKinAssignWarps + w;
    double loss = 0.0;
    if (p < a.P) {
        const int k0 = a.part_offsets[p], k1 = a.part_offsets[p + 1];
        const float s = 2.0f * a.lambda;
        float acc[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) acc[k] = 0.f;
        for (int k = k0 + lane; k < k1; k += 32) {
            const int i = a.sample_order[k];
            const int64_t si = a.src_idx[i];
            const int j = a.col4row[(int64_t)t * a.n + i];
            const float* sp = a.skinned + ((int64_t)t * a.N + si) * 3;
            const float* tp = a.tgt + ((int64_t)t * a.n + (j >= 0 ? j : 0)) * 3;
            const float* x = a.cano + si * 3;
            const float dx = sp[0] - tp[0], dy = sp[1] - tp[1], dz = sp[2] - tp[2];
            loss += (double)(dx * dx + dy * dy + dz * dz);
            const float g[3] = {s * dx, s * dy, s * dz};
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                acc[3 * r] += g[r] * x[0]; acc[3 * r + 1] += g[r] * x[1]; acc[3 * r + 2] += g[r] * x[2];
                acc[9 + r] += g[r];
            }
        }
#pragma unroll
        for (int k = 0; k < 12; ++k)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
        const int64_t tp = (int64_t)t * a.P + p;
        if (lane < 12 && (k1 > k0 || !a.accumulate)) {          // a part without samples keeps its gradient (or gets zeros)
            float v = 0.f;
#pragma unroll
            for (int k = 0; k < 12; ++k) v = lane == k ? acc[k] : v;
            float* o = lane < 9 ? a.gR + tp * 9 + lane : a.gtr + tp * 3 + (lane - 9);
            *o = a.accumulate ? *o + v : v;
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
        for (int q = 0; q < kKinAssignWarps; ++q) c += s_loss[q];
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

int launch_kin_assign(const KinAssign& a, cudaStream_t stream) {
    if (a.T <= 0) return kOk;
    if (a.P <= 0 || a.P > 32) return kErrUnsupported;
    dim3 grid((unsigned)a.T, (unsigned)ceil_div(a.P, kKinAssignWarps));
    kin_assign_kernel<<<grid, 32 * kKinAssignWarps, 0, stream>>>(a);
    REART_CHECK_LAUNCH();
    return kOk;
}

// ============================================================================================ flow loss
// The flow loss of run_robot.py:194-213 (networks/loss.py:10-21) and its gradient w.r.t. the poses, on a window of K
// consecutive frames of the complete sequence.  With one-hot skinning weights, slot s holding local frame t:
//   pred_k = win[k+1] - win[k],  err_k = pred_k - tflow[k],  d_k = d flow_loss / d pred_k (per point, per component):
//     mask set: 2 err (plain) | err if |err| < 1 else sign(err) (robust);  mask clear: 2 * 0.01 * pred
//   g = lambda (d_{s-1} - d_s)  (a term outside the window is dropped);  gR[t,p] += sum g x^T,  gtr[t,p] += sum g.
// One CTA per (slot, part): thread j takes the part's points j, j+256, ... (point_order groups them by part), then a fixed
// xor tree per warp and the warps in order.  Pair k's loss is counted (if q0 <= k < q1) by the units of slot k+1 when
// that slot is local, else of slot k.  The loss: per-CTA partials added in index order by the last CTA (ticket).
// flow_term_grad (flow_device.cuh) is the per-component rule, shared with flow_grad_kernel (flow.cu).
constexpr int kKinFlowThreads = 256;

int64_t kin_flow_blocks(int64_t K, int64_t P) { return K * P; }

__global__ void __launch_bounds__(kKinFlowThreads) kin_flow_kernel(const KinFlow a) {
    constexpr int kWarps = kKinFlowThreads / 32;
    __shared__ float s_acc[kWarps][12];
    __shared__ double s_loss[kWarps];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int s = blockIdx.x, p = blockIdx.y, K = a.K;
    const int t = a.slot_frame[s];
    double loss = 0.0;
    const bool local = t >= 0 && t < a.T;
    const int k0 = a.part_offsets[p], k1 = a.part_offsets[p + 1];
    if (local && k1 > k0) {
        // which of the two adjacent pairs this unit counts the loss of
        const bool has_prev = s > 0, has_next = s < K - 1;
        const bool count_prev = has_prev && s - 1 >= a.q0 && s - 1 < a.q1;           // slot s is the pair's second slot
        const bool count_next = has_next && s >= a.q0 && s < a.q1 && a.slot_frame[s + 1] < 0;
        const int64_t N = a.N;
        float acc[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) acc[k] = 0.f;
        for (int k = k0 + threadIdx.x; k < k1; k += kKinFlowThreads) {
            const int64_t i = a.point_order[k];
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
            const float* x = a.cano + i * 3;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const float gr = a.lambda * g[r];
                acc[3 * r] += gr * x[0]; acc[3 * r + 1] += gr * x[1]; acc[3 * r + 2] += gr * x[2];
                acc[9 + r] += gr;
            }
        }
#pragma unroll
        for (int k = 0; k < 12; ++k)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
        if (lane == 0)
#pragma unroll
            for (int k = 0; k < 12; ++k) s_acc[w][k] = acc[k];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, o);
    if (lane == 0) s_loss[w] = loss;
    __syncthreads();
    if (local && threadIdx.x < 12 && (k1 > k0 || !a.accumulate)) {   // a part without points keeps its gradient (or gets zeros)
        float v = 0.f;
        if (k1 > k0)
            for (int q = 0; q < kWarps; ++q) v += s_acc[q][threadIdx.x];
        const int64_t tp = (int64_t)t * a.P + p;
        float* o = threadIdx.x < 9 ? a.gR + tp * 9 + threadIdx.x : a.gtr + tp * 3 + (threadIdx.x - 9);
        *o = a.accumulate ? *o + v : v;
    }
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

int launch_kin_flow(const KinFlow& a, cudaStream_t stream) {
    if (a.T <= 0) return kOk;
    if (a.P <= 0 || a.P > 32) return kErrUnsupported;
    if (a.K < 2) return kErrInvalidArg;
    dim3 grid((unsigned)a.K, (unsigned)a.P);
    kin_flow_kernel<<<grid, kKinFlowThreads, 0, stream>>>(a);
    REART_CHECK_LAUNCH();
    return kOk;
}

}  // namespace reart
