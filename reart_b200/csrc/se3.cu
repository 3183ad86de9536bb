// se3.cu -- fused SE(3) helpers of the hot path: 6D -> R, screw -> exp -> 4x4, tree forward kinematics,
// each with an analytic backward obtained by forward-mode dual numbers inside the kernel.
//
// Replaces (file:line under the reference tree)
//   screw_se3/geo_utils.py:632-651   rotation_6d_to_matrix
//   screw_se3/screw_utils.py:6-23    screw_param_to_exponential_coordinates
//   screw_se3/screw_utils.py:27-30   transform_from_exponential_coordinates
//   screw_se3/geo_utils.py:90-222    _so3_exp_map / _se3_V_matrix / se3_exp_map
//   utils/kinematic_utils.py:151-198 fk   (a Python double loop issuing ~10.5k ATen ops per fwd+bwd, SURVEY fact 7)
// reproducing the reference's numerical quirks (SURVEY Q8-Q10, Q17): strict |theta|<1e-6 / |theta-pi|<1e-6
// no-rot branch that ignores d; theta^2 |l|^2 clamped at 1e-4 (gradient of the clamp is 0 below it);
// axes are never normalised.
//
// These kernels are launch-latency bound (T*P elements); one thread per frame walks the tree.
#include "common.cuh"
#include "kernels.h"
#include "se3_device.cuh"
#include <algorithm>

namespace reart {

__global__ void rot6d_fwd_kernel(const float* __restrict__ d6, int64_t B, float* __restrict__ R) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= B) return;
    float in[6], out[9];
    for (int k = 0; k < 6; ++k) in[k] = d6[i * 6 + k];
    rot6d_eval<float>(in, out);
    for (int k = 0; k < 9; ++k) R[i * 9 + k] = out[k];
}

__global__ void rot6d_bwd_kernel(const float* __restrict__ d6, const float* __restrict__ gR, int64_t B,
                                 float* __restrict__ gd6) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= B) return;
    Dual<6> in[6], out[9];
    for (int k = 0; k < 6; ++k) in[k] = Dual<6>::var(d6[i * 6 + k], k);
    rot6d_eval<Dual<6>>(in, out);
    float g[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int o = 0; o < 9; ++o) {
        const float go = gR[i * 9 + o];
        for (int k = 0; k < 6; ++k) g[k] += go * out[o].d[k];
    }
    for (int k = 0; k < 6; ++k) gd6[i * 6 + k] = g[k];
}

int launch_rot6d_fwd(const float* d6, int64_t B, float* R, cudaStream_t stream) {
    if (B <= 0) return kOk;
    rot6d_fwd_kernel<<<(unsigned)ceil_div(B, 128), 128, 0, stream>>>(d6, B, R);
    REART_CHECK_LAUNCH();
    return kOk;
}
int launch_rot6d_bwd(const float* d6, const float* gR, int64_t B, float* gd6, cudaStream_t stream) {
    if (B <= 0) return kOk;
    rot6d_bwd_kernel<<<(unsigned)ceil_div(B, 64), 64, 0, stream>>>(d6, gR, B, gd6);
    REART_CHECK_LAUNCH();
    return kOk;
}

// ----------------------------------------------------------------------------- screw -> 4x4
__global__ void screw_fwd_kernel(const float* __restrict__ l, const float* __restrict__ m,
                                 const float* __restrict__ theta, const float* __restrict__ d, int64_t B,
                                 float* __restrict__ M) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= B) return;
    float L[3] = {l[3 * i], l[3 * i + 1], l[3 * i + 2]}, Mo[3] = {m[3 * i], m[3 * i + 1], m[3 * i + 2]}, out[12];
    screw_eval<float>(L, Mo, theta[i], d[i], out);
    for (int k = 0; k < 12; ++k) M[16 * i + k] = out[k];
    M[16 * i + 12] = 0.f; M[16 * i + 13] = 0.f; M[16 * i + 14] = 0.f; M[16 * i + 15] = 1.f;
}

__global__ void screw_bwd_kernel(const float* __restrict__ l, const float* __restrict__ m,
                                 const float* __restrict__ theta, const float* __restrict__ d,
                                 const float* __restrict__ gM, int64_t B, float* __restrict__ gl,
                                 float* __restrict__ gm, float* __restrict__ gtheta, float* __restrict__ gd) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= B) return;
    Dual<8> L[3], Mo[3], out[12];
    for (int k = 0; k < 3; ++k) { L[k] = Dual<8>::var(l[3 * i + k], k); Mo[k] = Dual<8>::var(m[3 * i + k], 3 + k); }
    screw_eval<Dual<8>>(L, Mo, Dual<8>::var(theta[i], 6), Dual<8>::var(d[i], 7), out);
    float g[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int o = 0; o < 12; ++o) {
        const float go = gM[16 * i + o];
        for (int k = 0; k < 8; ++k) g[k] += go * out[o].d[k];
    }
    for (int k = 0; k < 3; ++k) { gl[3 * i + k] = g[k]; gm[3 * i + k] = g[3 + k]; }
    gtheta[i] = g[6];
    gd[i] = g[7];
}

int launch_screw_fwd(const float* l, const float* m, const float* theta, const float* d, int64_t B, float* M,
                     cudaStream_t stream) {
    if (B <= 0) return kOk;
    screw_fwd_kernel<<<(unsigned)ceil_div(B, 128), 128, 0, stream>>>(l, m, theta, d, B, M);
    REART_CHECK_LAUNCH();
    return kOk;
}
int launch_screw_bwd(const float* l, const float* m, const float* theta, const float* d, const float* gM, int64_t B,
                     float* gl, float* gm, float* gtheta, float* gd, cudaStream_t stream) {
    if (B <= 0) return kOk;
    screw_bwd_kernel<<<(unsigned)ceil_div(B, 64), 64, 0, stream>>>(l, m, theta, d, gM, B, gl, gm, gtheta, gd);
    REART_CHECK_LAUNCH();
    return kOk;
}

// ----------------------------------------------------------------------------- forward kinematics
// one thread per frame; out [T,P,4,4] indexed by part id
__global__ void fk_fwd_kernel(const FkParams p, float* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.T) return;
    for (int oi = 0; oi < p.P; ++oi) {
        const int c = p.order[oi];
        float* M = out + ((int64_t)t * p.P + c) * 16;
        const int par = p.parent[c];
        if (par < 0) {
            for (int k = 0; k < 16; ++k) M[k] = (k % 5 == 0) ? 1.f : 0.f;
            continue;
        }
        const int e = p.edge[c];
        float th, dd; bool tv, dv;
        fk_joint_inputs(p, t, e, th, dd, tv, dv);
        float L[3] = {p.axis[3 * e], p.axis[3 * e + 1], p.axis[3 * e + 2]};
        float Mo[3] = {p.moment[3 * e], p.moment[3 * e + 1], p.moment[3 * e + 2]};
        float rel[12], res[12];
        screw_eval<float>(L, Mo, th, dd, rel);
        mat34_mul(out + ((int64_t)t * p.P + par) * 16, rel, res);
        for (int k = 0; k < 12; ++k) M[k] = res[k];
        M[12] = 0.f; M[13] = 0.f; M[14] = 0.f; M[15] = 1.f;
    }
}

// Backward.  gwork [T,P,4,4] holds dL/d fk on entry (a scratch COPY: it is accumulated into in place).
// g_axis/g_moment [E,3] (+= over frames, zero on entry), g_theta/g_dist [T,E] (zero on entry; g_dist may be null).
__global__ void fk_bwd_kernel(const FkParams p, const float* __restrict__ fk, float* __restrict__ gwork,
                              float* __restrict__ g_axis, float* __restrict__ g_moment, float* __restrict__ g_theta,
                              float* __restrict__ g_dist) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.T) return;
    const int E = p.P - 1;
    for (int oi = p.P - 1; oi >= 0; --oi) {                   // leaves first
        const int c = p.order[oi];
        const int par = p.parent[c];
        if (par < 0) continue;
        const int e = p.edge[c];
        float th, dd; bool tv, dv;
        fk_joint_inputs(p, t, e, th, dd, tv, dv);
        Dual<8> L[3], Mo[3], rel[12];
        for (int k = 0; k < 3; ++k) { L[k] = Dual<8>::var(p.axis[3 * e + k], k); Mo[k] = Dual<8>::var(p.moment[3 * e + k], 3 + k); }
        screw_eval<Dual<8>>(L, Mo, Dual<8>::var(th, 6), Dual<8>::var(dd, 7), rel);
        const float* A = fk + ((int64_t)t * p.P + par) * 16;  // parent pose
        float* G = gwork + ((int64_t)t * p.P + c) * 16;       // dL/d fk[c] (complete: children were folded already)
        float* Gp = gwork + ((int64_t)t * p.P + par) * 16;
        // dL/dTrel = A^T G  (top 3 rows), and  Gp += G Trel^T
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
        for (int k = 0; k < 3; ++k) { atomicAdd(g_axis + 3 * e + k, g8[k]); atomicAdd(g_moment + 3 * e + k, g8[3 + k]); }
        if (tv) g_theta[(int64_t)t * E + e] = g8[6];
        if (dv && g_dist) g_dist[(int64_t)t * E + e] = g8[7];
    }
}

int launch_fk_fwd(const FkParams& p, float* out, cudaStream_t stream) {
    if (p.T <= 0 || p.P <= 0) return kOk;
    fk_fwd_kernel<<<(unsigned)ceil_div(p.T, 32), 32, 0, stream>>>(p, out);
    REART_CHECK_LAUNCH();
    return kOk;
}

int launch_fk_bwd(const FkParams& p, const float* fk, const float* g_out, float* gwork, float* g_axis, float* g_moment,
                  float* g_theta, float* g_dist, cudaStream_t stream) {
    const int64_t E = p.P - 1;
    if (p.T <= 0 || p.P <= 0) return kOk;
    if (cudaMemcpyAsync(gwork, g_out, sizeof(float) * (size_t)p.T * p.P * 16, cudaMemcpyDeviceToDevice, stream) != cudaSuccess)
        return kErrLaunch;
    if (E > 0) {
        if (cudaMemsetAsync(g_axis, 0, sizeof(float) * (size_t)E * 3, stream) != cudaSuccess) return kErrLaunch;
        if (cudaMemsetAsync(g_moment, 0, sizeof(float) * (size_t)E * 3, stream) != cudaSuccess) return kErrLaunch;
        if (cudaMemsetAsync(g_theta, 0, sizeof(float) * (size_t)p.T * E, stream) != cudaSuccess) return kErrLaunch;
        if (g_dist && cudaMemsetAsync(g_dist, 0, sizeof(float) * (size_t)p.T * E, stream) != cudaSuccess) return kErrLaunch;
    }
    fk_bwd_kernel<<<(unsigned)ceil_div(p.T, 32), 32, 0, stream>>>(p, fk, gwork, g_axis, g_moment, g_theta, g_dist);
    REART_CHECK_LAUNCH();
    return kOk;
}

}  // namespace reart
