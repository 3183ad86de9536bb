// se3_device.cuh -- forward-mode dual numbers, 6D -> R, screw -> 3x4 and the forward-kinematics pieces shared by se3.cu,
// relax.cu and kin.cu.
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace reart {

// ----------------------------------------------------------------------------- forward-mode duals
template <int ND>
struct Dual {
    float v;
    float d[ND];
    __device__ Dual() {}
    __device__ explicit Dual(float c) : v(c) {
#pragma unroll
        for (int i = 0; i < ND; ++i) d[i] = 0.f;
    }
    __device__ static Dual var(float c, int k) {
        Dual r(c);
        r.d[k] = 1.f;
        return r;
    }
};
template <int ND>
__device__ __forceinline__ Dual<ND> operator+(const Dual<ND>& a, const Dual<ND>& b) {
    Dual<ND> r; r.v = a.v + b.v;
#pragma unroll
    for (int i = 0; i < ND; ++i) r.d[i] = a.d[i] + b.d[i];
    return r;
}
template <int ND>
__device__ __forceinline__ Dual<ND> operator-(const Dual<ND>& a, const Dual<ND>& b) {
    Dual<ND> r; r.v = a.v - b.v;
#pragma unroll
    for (int i = 0; i < ND; ++i) r.d[i] = a.d[i] - b.d[i];
    return r;
}
template <int ND>
__device__ __forceinline__ Dual<ND> operator-(const Dual<ND>& a) {
    Dual<ND> r; r.v = -a.v;
#pragma unroll
    for (int i = 0; i < ND; ++i) r.d[i] = -a.d[i];
    return r;
}
template <int ND>
__device__ __forceinline__ Dual<ND> operator*(const Dual<ND>& a, const Dual<ND>& b) {
    Dual<ND> r; r.v = a.v * b.v;
#pragma unroll
    for (int i = 0; i < ND; ++i) r.d[i] = a.d[i] * b.v + a.v * b.d[i];
    return r;
}
template <int ND>
__device__ __forceinline__ Dual<ND> operator*(const Dual<ND>& a, float s) {
    Dual<ND> r; r.v = a.v * s;
#pragma unroll
    for (int i = 0; i < ND; ++i) r.d[i] = a.d[i] * s;
    return r;
}
template <int ND>
__device__ __forceinline__ Dual<ND> operator/(const Dual<ND>& a, const Dual<ND>& b) {
    Dual<ND> r; r.v = a.v / b.v;
    const float inv = 1.0f / b.v;
#pragma unroll
    for (int i = 0; i < ND; ++i) r.d[i] = (a.d[i] - r.v * b.d[i]) * inv;
    return r;
}
template <int ND>
__device__ __forceinline__ Dual<ND> dsin(const Dual<ND>& a) {
    Dual<ND> r; r.v = sinf(a.v);
    const float c = cosf(a.v);
#pragma unroll
    for (int i = 0; i < ND; ++i) r.d[i] = c * a.d[i];
    return r;
}
template <int ND>
__device__ __forceinline__ Dual<ND> dcos(const Dual<ND>& a) {
    Dual<ND> r; r.v = cosf(a.v);
    const float s = -sinf(a.v);
#pragma unroll
    for (int i = 0; i < ND; ++i) r.d[i] = s * a.d[i];
    return r;
}
template <int ND>
__device__ __forceinline__ Dual<ND> dsqrt(const Dual<ND>& a) {
    Dual<ND> r; r.v = sqrtf(a.v);
    const float k = r.v > 0.f ? 0.5f / r.v : 0.f;            // torch: d sqrt / norm at 0 -> 0 subgradient
#pragma unroll
    for (int i = 0; i < ND; ++i) r.d[i] = k * a.d[i];
    return r;
}
// torch.clamp(x, min=lo): passes the gradient where x >= lo, zero below
template <int ND>
__device__ __forceinline__ Dual<ND> dclamp_min(const Dual<ND>& a, float lo) {
    if (a.v >= lo) return a;
    return Dual<ND>(lo);
}
// plain-float overloads so the same templated code serves the forward-only kernels
__device__ __forceinline__ float dsin(float a) { return sinf(a); }
__device__ __forceinline__ float dcos(float a) { return cosf(a); }
__device__ __forceinline__ float dsqrt(float a) { return sqrtf(a); }
__device__ __forceinline__ float dclamp_min(float a, float lo) { return a >= lo ? a : lo; }

template <typename S> __device__ __forceinline__ S lit(float c);
template <> __device__ __forceinline__ float lit<float>(float c) { return c; }
template <> __device__ __forceinline__ Dual<6> lit<Dual<6>>(float c) { return Dual<6>(c); }
template <> __device__ __forceinline__ Dual<8> lit<Dual<8>>(float c) { return Dual<8>(c); }
__device__ __forceinline__ float val(float a) { return a; }
template <int ND> __device__ __forceinline__ float val(const Dual<ND>& a) { return a.v; }

// ----------------------------------------------------------------------------- 6D -> R
// F.normalize(v, eps=1e-12): v / max(|v|, eps)
template <typename S>
__device__ __forceinline__ void normalize3(const S* v, S* o) {
    S n = dsqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
    S den = dclamp_min(n, 1e-12f);
    o[0] = v[0] / den; o[1] = v[1] / den; o[2] = v[2] / den;
}
template <typename S>
__device__ __forceinline__ void rot6d_eval(const S* d6, S* R) {
    S b1[3], b2[3], u[3];
    normalize3(d6, b1);
    S dot = b1[0] * d6[3] + b1[1] * d6[4] + b1[2] * d6[5];
    for (int k = 0; k < 3; ++k) u[k] = d6[3 + k] - dot * b1[k];
    normalize3(u, b2);
    R[0] = b1[0]; R[1] = b1[1]; R[2] = b1[2];
    R[3] = b2[0]; R[4] = b2[1]; R[5] = b2[2];
    R[6] = b1[1] * b2[2] - b1[2] * b2[1];
    R[7] = b1[2] * b2[0] - b1[0] * b2[2];
    R[8] = b1[0] * b2[1] - b1[1] * b2[0];
}


// ----------------------------------------------------------------------------- screw -> 4x4
// M (row-major 3x4: [R | t]) from (l, m, theta, d): screw_se3/screw_utils.py:6-30 over geo_utils.py:90-222, with the
// reference's quirks (se3.cu header)
template <typename S>
__device__ __forceinline__ void screw_eval(const S* l, const S* m, const S& theta, const S& d, S* M) {
    const float eps = 1e-6f;
    const float pi_f = 3.14159265358979323846f;
    const float th = val(theta);
    const bool no_rot = (fabsf(th) < eps) || (fabsf(th - pi_f) < eps);
    S w[3], v[3];
    if (!no_rot) {
        S q[3] = {l[1] * m[2] - l[2] * m[1], l[2] * m[0] - l[0] * m[2], l[0] * m[1] - l[1] * m[0]};
        S h = d / theta;
        S c[3] = {q[1] * l[2] - q[2] * l[1], q[2] * l[0] - q[0] * l[2], q[0] * l[1] - q[1] * l[0]};
        for (int k = 0; k < 3; ++k) { w[k] = l[k] * theta; v[k] = (c[k] + h * l[k]) * theta; }
    } else {
        for (int k = 0; k < 3; ++k) { w[k] = lit<S>(0.f) * theta; v[k] = l[k] * theta; }
    }
    S nrm = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
    S ang = dsqrt(dclamp_min(nrm, 1e-4f));
    S one = lit<S>(1.0f);
    S inv = one / ang;
    S sn = dsin(ang), cs = dcos(ang);
    S fac1 = inv * sn;
    S fac2 = inv * inv * (one - cs);
    S facV1 = (one - cs) / (ang * ang);
    S facV2 = (ang - sn) / (ang * ang * ang);
    S zero = lit<S>(0.f);
    S K[9] = {zero, -w[2], w[1], w[2], zero, -w[0], -w[1], w[0], zero};
    S K2[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) K2[3 * i + j] = K[3 * i] * K[j] + K[3 * i + 1] * K[3 + j] + K[3 * i + 2] * K[6 + j];
    for (int i = 0; i < 3; ++i) {
        S Vr[3];
        for (int j = 0; j < 3; ++j) {
            S I = lit<S>(i == j ? 1.f : 0.f);
            M[4 * i + j] = fac1 * K[3 * i + j] + fac2 * K2[3 * i + j] + I;
            Vr[j] = I + K[3 * i + j] * facV1 + K2[3 * i + j] * facV2;
        }
        M[4 * i + 3] = Vr[0] * v[0] + Vr[1] * v[1] + Vr[2] * v[2];
    }
}

// ----------------------------------------------------------------------------- forward kinematics (tree walk pieces)
__device__ __forceinline__ void mat34_mul(const float* A, const float* Bm, float* C) {   // [A;0001]*[B;0001], 3x4 blocks
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 4; ++j) {
            float s = A[4 * i] * Bm[j] + A[4 * i + 1] * Bm[4 + j] + A[4 * i + 2] * Bm[8 + j];
            if (j == 3) s += A[4 * i + 3];
            C[4 * i + j] = s;
        }
    }
}

__device__ __forceinline__ void fk_joint_inputs(const FkParams& p, int t, int e, float& th, float& dd, bool& th_var,
                                                bool& d_var) {
    const int E = p.P - 1;
    const int jt = p.joint_type ? p.joint_type[e] : 0;
    th = p.theta[(int64_t)t * E + e];
    th_var = true;
    d_var = p.distance != nullptr;
    dd = d_var ? p.distance[(int64_t)t * E + e] : 1e-6f;
    if (jt == 1) { dd = 1e-6f; d_var = false; }              // revolute  (kinematic_utils.py:181-184)
    if (jt == 2) { th = 1e-6f; th_var = false; }             // prismatic (kinematic_utils.py:176-179)
}

}  // namespace reart
