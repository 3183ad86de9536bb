// lap.cu -- the assignment loss on the GPU: exact linear-sum-assignment per frame + the matched-pair loss/gradient.
//
// Replaces the refresh block of run_robot.py:164-187 (run_real.py:180-203, run_sapien.py:179-203):
//   cost = torch.cdist(pc_src, pc_tgt).cpu().numpy();  indices = [linear_sum_assignment(c) for c in cost]
// (utils/model_utils.py:85-89 when --use_nproc: a multiprocessing.Pool spawned per refresh), i.e. a D2H copy of T n x n
// matrices and T Hungarian solves on the host every `assign_gap` iterations, and of utils/model_utils.py:92-103
// (compute_ass_err).  Here: one CTA per frame runs the same algorithm scipy does -- shortest augmenting paths with
// dual variables (Jonker-Volgenant as in scipy/optimize/rectangular_lsap) -- so the result is an exactly optimal
// assignment of the float32 Euclidean costs, with
//   * costs formed on the fly from the sample points (no n x n matrix, no D2H, graph-capturable);
//   * every thread owning 4 columns in REGISTERS (target point, dual v, current shortest path cost), so one Dijkstra
//     step is 4 cost evaluations + one block-wide arg-min (two shuffle trees, ONE barrier);
//   * dual variables and path costs in float64 like scipy; the arg-min order is (cost, unassigned first, lowest column);
//   * a column-reduction start (v_j = min_i c_ij, each column's arg-min row taken greedily, lowest column first):
//     dual feasible and tight, typically assigns about half the rows before the first augmentation.
// n <= 4096 samples per frame (the reference's n is N / downsample = 1024; its own model-selection term uses n = N = 4096).
#include "common.cuh"
#include "kernels.h"
#include <algorithm>

namespace reart {

constexpr int kLapCols = 4;                                  // columns per thread

struct LapCand {
    u64 d;                                                   // order-preserving image of the path cost (double)
    unsigned t;                                              // (assigned ? 1 : 0) << 31 | column
};
__device__ __forceinline__ bool lap_better(const LapCand& a, const LapCand& b) {
    return a.d < b.d || (a.d == b.d && a.t < b.t);
}
__device__ __forceinline__ u64 lap_order_bits(double v) {
    const u64 b = (u64)__double_as_longlong(v);
    return b ^ ((b >> 63) ? ~0ull : 0x8000000000000000ull);
}
__device__ __forceinline__ double lap_from_bits(u64 k) {
    const u64 b = (k >> 63) ? (k ^ 0x8000000000000000ull) : ~k;
    return __longlong_as_double((long long)b);
}
__device__ __forceinline__ LapCand lap_warp_min(LapCand c) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        LapCand o;
        o.d = __shfl_xor_sync(0xffffffffu, c.d, s);
        o.t = __shfl_xor_sync(0xffffffffu, c.t, s);
        if (lap_better(o, c)) c = o;
    }
    return c;
}
__device__ __forceinline__ float lap_cost(const float4& s, float tx, float ty, float tz) {
    return sqrtf(sqdist_scalar(s.x, s.y, s.z, tx, ty, tz));
}

// src_base [B, src_stride/3 points, 3] read through src_idx [n] (or densely when src_idx is null); tgt [B,n,3].
template <int NT>
__global__ void __launch_bounds__(NT) lap_jv_kernel(const float* __restrict__ src_base, const int64_t* __restrict__ src_idx,
                                                    int64_t src_stride, const float* __restrict__ tgt, int n,
                                                    int* __restrict__ col4row_out, double* __restrict__ total_out,
                                                    double* __restrict__ dual_u, int warm) {
    extern __shared__ __align__(16) unsigned char lap_sm[];
    float4* s_src = reinterpret_cast<float4*>(lap_sm);                      // [n]
    double* s_short = reinterpret_cast<double*>(s_src + n);                 // [n]
    double* s_u = s_short + n;                                              // [n]
    int* s_path = reinterpret_cast<int*>(s_u + n);                          // [n]
    int* s_row4col = s_path + n;                                            // [n]
    int* s_col4row = s_row4col + n;                                         // [n]
    int* s_sr = s_col4row + n;                                              // [n] rows visited by the current search
    __shared__ LapCand s_red[2][NT / 32];
    __shared__ double s_tot[NT / 32];
    constexpr int NW = NT / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.x;
    const float* __restrict__ sb = src_base + (int64_t)b * src_stride;
    const float* __restrict__ tb = tgt + (int64_t)b * n * 3;

    for (int i = tid; i < n; i += NT) {
        const int64_t si = src_idx ? src_idx[i] : (int64_t)i;
        s_src[i] = make_float4(sb[3 * si], sb[3 * si + 1], sb[3 * si + 2], 0.f);
        s_u[i] = (dual_u && warm) ? dual_u[(int64_t)b * n + i] : 0.0;      // warm start: the previous solve's row duals
        s_col4row[i] = 0x7fffffff;
        s_row4col[i] = -1;
    }
    float tx[kLapCols], ty[kLapCols], tz[kLapCols];
    double v[kLapCols], sh[kLapCols];
    bool valid[kLapCols];
#pragma unroll
    for (int k = 0; k < kLapCols; ++k) {
        const int j = tid + k * NT;
        valid[k] = j < n;
        tx[k] = valid[k] ? tb[3 * j] : 0.f; ty[k] = valid[k] ? tb[3 * j + 1] : 0.f; tz[k] = valid[k] ? tb[3 * j + 2] : 0.f;
        v[k] = 0.0; sh[k] = 0.0;
    }
    __syncthreads();

    // ---- column reduction: v_j = min_i (c_ij - u_i) (first arg-min row), greedy assignment of those tight edges, lowest
    // column wins a contested row.  Any u is admissible (reduced costs end up >= 0 with one tight row per column).  With
    // u = 0 this is the classic start; with the previous refresh's duals (the clouds moved by a few optimiser steps) nearly
    // every column finds its old partner again and almost no augmentation is left.
    int argrow[kLapCols];
    {
        double best[kLapCols];
#pragma unroll
        for (int k = 0; k < kLapCols; ++k) { best[k] = INFINITY; argrow[k] = 0; }
        for (int i = 0; i < n; ++i) {
            const float4 s = s_src[i];
            const double ui = s_u[i];
#pragma unroll
            for (int k = 0; k < kLapCols; ++k) {
                const double c = (double)lap_cost(s, tx[k], ty[k], tz[k]) - ui;
                if (c < best[k]) { best[k] = c; argrow[k] = i; }
            }
        }
#pragma unroll
        for (int k = 0; k < kLapCols; ++k)
            if (valid[k]) { v[k] = best[k]; atomicMin(&s_col4row[argrow[k]], tid + k * NT); }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kLapCols; ++k)
        if (valid[k] && s_col4row[argrow[k]] == tid + k * NT) s_row4col[tid + k * NT] = argrow[k];
    __syncthreads();
    for (int i = tid; i < n; i += NT)
        if (s_col4row[i] == 0x7fffffff) s_col4row[i] = -1;
    __syncthreads();

    // ---- one shortest augmenting path per free row (scipy rectangular_lsap: augmenting_path + dual update + augment)
    unsigned parity = 0;
    for (int cur = 0; cur < n; ++cur) {
        if (s_col4row[cur] >= 0) continue;                               // block-uniform
        unsigned sc = 0u, assigned = 0u;
#pragma unroll
        for (int k = 0; k < kLapCols; ++k) {
            sh[k] = INFINITY;
            if (valid[k] && s_row4col[tid + k * NT] >= 0) assigned |= 1u << k;
        }
        int nsr = 0, i = cur, sink = -1;
        double minval = 0.0;
        while (sink < 0) {
            if (tid == 0) s_sr[nsr] = i;
            ++nsr;
            const float4 s = s_src[i];
            const double ui = s_u[i];
            LapCand best;
            best.d = ~0ull; best.t = ~0u;
#pragma unroll
            for (int k = 0; k < kLapCols; ++k) {
                if (valid[k] && !((sc >> k) & 1u)) {
                    const double r = minval + (double)lap_cost(s, tx[k], ty[k], tz[k]) - ui - v[k];
                    if (r < sh[k]) { sh[k] = r; s_path[tid + k * NT] = i; }
                    LapCand c;
                    c.d = lap_order_bits(sh[k]);
                    c.t = (((assigned >> k) & 1u) << 31) | (unsigned)(tid + k * NT);
                    if (lap_better(c, best)) best = c;
                }
            }
            best = lap_warp_min(best);
            if (lane == 0) s_red[parity][warp] = best;
            __syncthreads();
            LapCand g;
            if (lane < NW) g = s_red[parity][lane];
            else { g.d = ~0ull; g.t = ~0u; }
            g = lap_warp_min(g);                                 // every warp reduces the NW slots itself: no second barrier
            parity ^= 1u;
            if (g.d == ~0ull && g.t == ~0u) { sink = -2; break; }       // no reachable column: cannot happen for finite costs
            const int jstar = (int)(g.t & 0x7fffffffu);
            minval = lap_from_bits(g.d);
            if (jstar % NT == tid) sc |= 1u << (jstar / NT);
            if (!(g.t >> 31)) sink = jstar;
            else i = s_row4col[jstar];
        }
        // duals (before the augmentation, with the pre-augmentation col4row), then flip the path
#pragma unroll
        for (int k = 0; k < kLapCols; ++k)
            if (valid[k]) s_short[tid + k * NT] = sh[k];
        __syncthreads();
        if (sink >= 0) {
            if (tid == 0) s_u[cur] += minval;
            for (int e = 1 + tid; e < nsr; e += NT) {
                const int r = s_sr[e];
                s_u[r] += minval - s_short[s_col4row[r]];
            }
#pragma unroll
            for (int k = 0; k < kLapCols; ++k)
                if ((sc >> k) & 1u) v[k] -= minval - sh[k];
        }
        __syncthreads();
        if (tid == 0 && sink >= 0) {
            int j = sink;
            for (;;) {
                const int r = s_path[j];
                s_row4col[j] = r;
                const int prev = s_col4row[r];
                s_col4row[r] = j;
                j = prev;
                if (r == cur) break;
            }
        }
        __syncthreads();
    }

    // ---- outputs: assignment, row duals for the next warm start, (optionally) the total cost in float64
    double part = 0.0;
    for (int i = tid; i < n; i += NT) {
        const int j = s_col4row[i];
        if (dual_u) dual_u[(int64_t)b * n + i] = s_u[i];
        col4row_out[(int64_t)b * n + i] = j;
        if (total_out && j >= 0) part += (double)lap_cost(s_src[i], tb[3 * j], tb[3 * j + 1], tb[3 * j + 2]);
    }
    if (total_out) {
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) part += __shfl_xor_sync(0xffffffffu, part, s);
        if (lane == 0) s_tot[warp] = part;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
            for (int w = 0; w < NW; ++w) t += s_tot[w];
            total_out[b] = t;
        }
    }
}

template <int NT>
static int launch_lap_nt(const float* src_base, const int64_t* src_idx, int64_t src_stride, const float* tgt, int64_t B,
                         int64_t n, int n_max, int* col4row, double* total, double* dual_u, int warm, cudaStream_t stream) {
    const size_t smem = (size_t)n * (16 + 8 + 8 + 4 * 4);
    static bool attr_done[64] = {};
    int devid = 0;
    cudaGetDevice(&devid);
    // static shared memory (reduction slots) comes on top of the dynamic part: opt in well below the 48 KB default limit.
    // smem grows with n, so the opt-in is made once per device for the bucket's LARGEST n: a later call with a larger n
    // than the first must not exceed what was opted in
    if (smem > 32 * 1024 && (devid < 0 || devid >= 64 || !attr_done[devid])) {
        const size_t smem_max = (size_t)n_max * (16 + 8 + 8 + 4 * 4);
        if (cudaFuncSetAttribute(lap_jv_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max) != cudaSuccess)
            return kErrUnsupported;
        if (devid >= 0 && devid < 64) attr_done[devid] = true;
    }
    lap_jv_kernel<NT><<<(unsigned)B, NT, smem, stream>>>(src_base, src_idx, src_stride, tgt, (int)n, col4row, total, dual_u,
                                                         warm);
    REART_CHECK_LAUNCH();
    return kOk;
}

int launch_lap(const float* src_base, const int64_t* src_idx, int64_t src_stride, const float* tgt, int64_t B, int64_t n,
               int* col4row, double* total, double* dual_u, int warm, cudaStream_t stream) {
    if (B <= 0 || n <= 0) return kOk;
    if (n > 4096) return kErrUnsupported;
    if (n <= 512) return launch_lap_nt<128>(src_base, src_idx, src_stride, tgt, B, n, 512, col4row, total, dual_u, warm, stream);
    if (n <= 1024) return launch_lap_nt<256>(src_base, src_idx, src_stride, tgt, B, n, 1024, col4row, total, dual_u, warm, stream);
    if (n <= 2048) return launch_lap_nt<512>(src_base, src_idx, src_stride, tgt, B, n, 2048, col4row, total, dual_u, warm, stream);
    return launch_lap_nt<1024>(src_base, src_idx, src_stride, tgt, B, n, 4096, col4row, total, dual_u, warm, stream);
}

// ---------------------------------------------------------------------------------------------- matched-pair loss
// loss += lambda * sum_{t,i} |skinned[t, src_idx[i]] - tgt[t, col4row[t,i]]|^2 ;  g_skinned[t, src_idx[i]] += 2 lambda (a - b)
// (run_robot.py:181-187).  FPS indices are distinct, so every skinned point is touched at most once per frame: plain
// read-modify-write, no atomics; the loss is summed by ONE block in a fixed order and added to *loss (single writer).
constexpr int kAssignThreads = 1024;
__global__ void __launch_bounds__(kAssignThreads) assign_loss_grad_kernel(const float* __restrict__ skinned,
                                                                          const int64_t* __restrict__ src_idx,
                                                                          const float* __restrict__ tgt,
                                                                          const int* __restrict__ col4row, int T, int N, int n,
                                                                          float lambda, float* __restrict__ g_skinned,
                                                                          int accumulate, double* __restrict__ loss) {
    __shared__ double s_w[kAssignThreads / 32];
    double part = 0.0;
    const int64_t total = (int64_t)T * n;
    for (int64_t e = threadIdx.x; e < total; e += kAssignThreads) {
        const int64_t t = e / n, i = e - t * n;
        const int64_t si = src_idx[i];
        const int j = col4row[e];
        const float* a = skinned + (t * N + si) * 3;
        const float* bpt = tgt + (t * n + (j >= 0 ? j : 0)) * 3;
        const float dx = a[0] - bpt[0], dy = a[1] - bpt[1], dz = a[2] - bpt[2];
        part += (double)(dx * dx + dy * dy + dz * dz);
        if (g_skinned) {
            float* g = g_skinned + (t * N + si) * 3;
            const float s = 2.0f * lambda;
            if (accumulate) { g[0] += s * dx; g[1] += s * dy; g[2] += s * dz; }
            else { g[0] = s * dx; g[1] = s * dy; g[2] = s * dz; }
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) part += __shfl_xor_sync(0xffffffffu, part, s);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tsum = 0.0;
        for (int w = 0; w < kAssignThreads / 32; ++w) tsum += s_w[w];
        *loss += (double)lambda * tsum;
    }
}

int launch_assign_loss_grad(const float* skinned, const int64_t* src_idx, const float* tgt, const int* col4row, int64_t T,
                            int64_t N, int64_t n, float lambda, float* g_skinned, int accumulate, double* loss,
                            cudaStream_t stream) {
    if (T <= 0 || n <= 0) return kOk;
    assign_loss_grad_kernel<<<1, kAssignThreads, 0, stream>>>(skinned, src_idx, tgt, col4row, (int)T, (int)N, (int)n, lambda,
                                                              g_skinned, accumulate, loss);
    REART_CHECK_LAUNCH();
    return kOk;
}

}  // namespace reart
