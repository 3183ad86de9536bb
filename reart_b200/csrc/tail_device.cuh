// tail_device.cuh -- the pieces every fused "tail" kernel (relax.cu, kin.cu) ends with: torch.optim.Adam on one element and
// the in-CTA one-shot all-reduce of a small gradient bucket over peer memory.
#pragma once
#include "common.cuh"

namespace reart {

// torch.optim.Adam (no amsgrad), one element: exp_avg.lerp_(g, 1-b1); exp_avg_sq.mul_(b2).addcmul_(g, g, 1-b2);
// p -= (lr / bc1) * exp_avg / (sqrt(exp_avg_sq) / sqrt(bc2) + eps)        (torch/optim/adam.py, _fused_adam math)
struct AdamCoef {
    float lr_over_bc1, inv_bc2_sqrt, b1, b2, eps, wd;
};
__device__ __forceinline__ void adam_update(float* p, float* m, float* v, float g, const AdamCoef& c) {
    const float pv = *p;
    if (c.wd != 0.f) g += c.wd * pv;
    const float mv = *m + (1.0f - c.b1) * (g - *m);
    const float vv = c.b2 * *v + (1.0f - c.b2) * g * g;
    *m = mv; *v = vv;
    *p = pv - c.lr_over_bc1 * mv / (sqrtf(vv) * c.inv_bc2_sqrt + c.eps);
}
__device__ __forceinline__ AdamCoef adam_coef(float lr, float b1, float b2, float eps, float wd, float step) {
    AdamCoef c;
    const double bc1 = 1.0 - pow((double)b1, (double)step), bc2 = 1.0 - pow((double)b2, (double)step);
    c.lr_over_bc1 = (float)((double)lr / bc1);
    c.inv_bc2_sqrt = (float)(1.0 / sqrt(bc2));
    c.b1 = b1; c.b2 = b2; c.eps = eps; c.wd = wd;
    return c;
}

__device__ __forceinline__ void st_release_sys_u32(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ld_volatile_f32_(const float* p) {
    float v;
    asm volatile("ld.volatile.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}

// In-CTA one-shot all-reduce of `bucket[0..n)` over peer memory: the protocol of allreduce_oneshot_kernel
// (allreduce.cu: stage in the symmetric buffer of parity `epoch+1`, flag every peer, wait for every flag, sum all
// ranks' buckets in rank order => identical bits everywhere).  Returns false if a peer never showed up.
__device__ inline bool cta_allreduce_oneshot(const unsigned long long* __restrict__ peer_base, int rank, int world, int n,
                                      int n_pad, unsigned* __restrict__ epoch, float* __restrict__ bucket, int* s_ok) {
    const unsigned e = *epoch + 1u;
    const int half = (int)(e & 1u);
    float* mine = reinterpret_cast<float*>(peer_base[rank]) + (size_t)half * n_pad;
    for (int i = threadIdx.x; i < n; i += blockDim.x) mine[i] = bucket[i];
    if (threadIdx.x == 0) *s_ok = 1;
    __syncthreads();
    if ((int)threadIdx.x < world) {
        __threadfence_system();
        unsigned* peer_flags = reinterpret_cast<unsigned*>(reinterpret_cast<float*>(peer_base[threadIdx.x]) + 2 * (size_t)n_pad);
        st_release_sys_u32(peer_flags + rank, e);
        const unsigned* my_flags = reinterpret_cast<const unsigned*>(reinterpret_cast<float*>(peer_base[rank]) + 2 * (size_t)n_pad);
        long long spins = 0;
        while ((int)(ld_acquire_sys_u32(my_flags + threadIdx.x) - e) < 0) {
            if (++spins > (1LL << 26)) { *s_ok = 0; break; }
        }
    }
    __syncthreads();
    const bool ok = *s_ok != 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float sum = 0.f;
        for (int r = 0; r < world; ++r)
            sum += ld_volatile_f32_(reinterpret_cast<const float*>(peer_base[r]) + (size_t)half * n_pad + i);
        bucket[i] = ok ? sum : __int_as_float(0x7fc00000);
    }
    __syncthreads();
    if (threadIdx.x == 0) *epoch = e;
    return ok;
}

}  // namespace reart
