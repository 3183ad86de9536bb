// energy.cu -- fused tail of the energy evaluation: from the (min, chunk) keys of the symmetric search
// to the loss and its gradient w.r.t. the skinned cloud.
//
// Fuses what the reference does in four steps: index recovery (inside chamferdist._C.knn_points_idx,
// utils/chamfer.py:174), torch.sum of the per-point distances (networks/loss.py:27-28) and the two
// _knn_points.backward calls (utils/chamfer.py:195-209):
//   loss   = sum_i d(src_i, tgt_nn(i)) + sum_j d(tgt_j, src_nn(j))
//   g_src  = gscale * [ 2 (src_i - tgt_nn(i))  -  sum_{j: nn(j)=i} 2 (tgt_j - src_i) ]
//
// Deterministic by construction (upstream's backward, and round 1 here, scatter with float atomics whose order changes
// from run to run):
//   * column pass first: every observed point recovers its arg-min source point and adds its term to a 64-bit
//     FIXED-POINT accumulator per (source point, axis).  The scale 2^k comes from a bound the search kernel leaves
//     behind (largest column minimum, common.cuh fixed_point_exponent), so no sum can overflow and every term keeps
//     >= 37 bits below its own magnitude; integer adds commute, so the result does not depend on atomic order;
//   * row pass second: direct term + converted accumulator, plain coalesced stores (no zero fill of g_src);
//   * loss: one double per block into a partials array, the last block to finish (ticket) adds them in index order.
// Memory-bound O(B (N+M)); both passes use the batched index recovery of common.cuh.
#include "common.cuh"
#include "kernels.h"
#include <algorithm>

namespace reart {

constexpr int kEnergyThreads = 256;

__device__ __forceinline__ double block_sum(double local, double* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = local;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 0; w < kEnergyThreads / 32; ++w) s += sh[w];
    }
    return s;
}

// ---- exact tie path of a search over permuted copies (EnergyParams row_order ...): the lowest caller index among the
// points `pts` [n,3] at exactly distance d from q -- what the brute force returns -- found by the whole warp, 512 points
// per round in caller order, stopping at the first round with a hit.  Only points whose tie word equals their minimum
// come here (two search chunks reach it); worst case (lattices, duplicates) one sweep of the other cloud per such point.
__device__ __forceinline__ int warp_lowest_match(const float* __restrict__ pts, int n, float qx, float qy, float qz, float d) {
    const int lane = threadIdx.x & 31;
    constexpr int kPer = 16;
    for (int j0 = 0; j0 < n; j0 += 32 * kPer) {
        int hit = 0x7fffffff;
#pragma unroll
        for (int u = kPer - 1; u >= 0; --u) {
            const int j = j0 + 32 * u + lane;
            if (j < n) {
                const float* t = pts + (int64_t)j * 3;
                if (sqdist_scalar(qx, qy, qz, __ldg(t), __ldg(t + 1), __ldg(t + 2)) == d) hit = j;
            }
        }
        hit = (int)__reduce_min_sync(0xffffffffu, (unsigned)hit);
        if (hit != 0x7fffffff) return hit;
    }
    return 0;                                                  // unreachable: d is a computed distance to one of the points
}

// Every flagged lane of the warp in turn: broadcast its query, resolve it with the whole warp.
__device__ __forceinline__ void resolve_flagged(bool flagged, const float* __restrict__ pts_b, int n, float qx, float qy,
                                                float qz, float d, int64_t b, int& idx, unsigned long long* count) {
    unsigned fl = __ballot_sync(0xffffffffu, flagged);
    if (fl && count && (threadIdx.x & 31) == 0) atomicAdd(count, (unsigned long long)__popc(fl));
    while (fl) {
        const int src = __ffs(fl) - 1;
        fl &= fl - 1;
        const float x = __shfl_sync(0xffffffffu, qx, src), y = __shfl_sync(0xffffffffu, qy, src);
        const float z = __shfl_sync(0xffffffffu, qz, src), dd = __shfl_sync(0xffffffffu, d, src);
        const int64_t bb = __shfl_sync(0xffffffffu, b, src);
        const int r = warp_lowest_match(pts_b + bb * (int64_t)n * 3, n, x, y, z, dd);
        if ((int)(threadIdx.x & 31) == src) idx = r;
    }
}

// ---- column pass: observed point j -> arg-min source point i, fixed-point scatter of -2 g (tgt_j - src_i)
// The loops run warp-uniformly (lane = f - f0) for the warp-wide tie path; every thread visits the same f as a plain
// grid-stride loop would, so the per-thread sums keep their association.
template <bool ORDERED>
__global__ void __launch_bounds__(kEnergyThreads) energy_cols_kernel(const EnergyParams p) {
    __shared__ double sh[kEnergyThreads / 32];
    const int64_t total = (int64_t)p.B * p.M;
    const float g2 = 2.0f * p.gscale;
    const float scale = ldexpf(1.0f, fixed_point_exponent(*p.col_bound, fabsf(g2), p.M));
    double local = 0.0;
    const int lane = threadIdx.x & 31;
    for (int64_t f0 = blockIdx.x * (int64_t)blockDim.x + (threadIdx.x - lane); f0 < total; f0 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t f = f0 + lane;
        const bool valid = f < total;
        int64_t b = 0, s = 0;
        float dmin = 0.f, ax = 0.f, ay = 0.f, az = 0.f;
        int i = 0;
        bool flagged = false;
        if (valid) {
            b = f / p.M;
            s = ORDERED ? b * p.M + p.tgt_inv[f] : f;            // the search's position of this point
            const u64 key = p.keys_b[s];
            dmin = __uint_as_float((unsigned)(key >> 32));
            const float* a = p.tgt + f * 3;
            ax = a[0]; ay = a[1]; az = a[2];
            flagged = ORDERED && p.tie_b[s] == (unsigned)(key >> 32);
            if (!flagged) {
                i = rescan_sorted_chunk_q(p.src_packed + b * (int64_t)p.n_pad * 3, p.src_perm + b * (int64_t)p.n_pad,
                                          p.src_xq + b * (int64_t)(p.n_pad / kSortedChunk) * kQuantiles,
                                          (unsigned)(key & 0xffffffffu), ax, ay, az, dmin);
                if (i >= p.N) i = 0;
                if (ORDERED) i = p.row_order[b * p.row_stride + i];
            }
        }
        if (ORDERED) resolve_flagged(flagged, p.src, p.N, ax, ay, az, dmin, b, i, p.ties);
        if (!valid) continue;
        const float* t = p.src + (b * p.N + i) * 3;
        unsigned long long* go = reinterpret_cast<unsigned long long*>(p.acc) + (b * p.N + i) * 3;
        // two's complement: adding the unsigned image of a negative term is the signed add
        atomicAdd(go + 0, (unsigned long long)__float2ll_rn(-g2 * (ax - t[0]) * scale));
        atomicAdd(go + 1, (unsigned long long)__float2ll_rn(-g2 * (ay - t[1]) * scale));
        atomicAdd(go + 2, (unsigned long long)__float2ll_rn(-g2 * (az - t[2]) * scale));
        local += (double)dmin;
        if (p.d_bwd) p.d_bwd[f] = dmin;
        if (p.i_bwd) p.i_bwd[f] = i;
        if (p.nn_cols) p.nn_cols[f] = i;                         // seeds by caller index
    }
    const double s = block_sum(local, sh);
    if (threadIdx.x == 0) p.partials[blockIdx.x] = s;
}

// ---- row pass: skinned point i -> arg-min observed point, g = direct term + accumulated reverse terms; final loss
template <bool ORDERED>
__global__ void __launch_bounds__(kEnergyThreads) energy_rows_kernel(const EnergyParams p, int col_blocks) {
    __shared__ double sh[kEnergyThreads / 32];
    __shared__ bool last;
    const int64_t total = (int64_t)p.B * p.N;
    const float g2 = 2.0f * p.gscale;
    const float inv = ldexpf(1.0f, -fixed_point_exponent(*p.col_bound, fabsf(g2), p.M));
    double local = 0.0;
    const int lane = threadIdx.x & 31;
    for (int64_t e0 = blockIdx.x * (int64_t)blockDim.x + (threadIdx.x - lane); e0 < total; e0 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = e0 + lane;
        const bool valid = e < total;
        int64_t b = 0, s = 0;
        float dmin = 0.f, ax = 0.f, ay = 0.f, az = 0.f;
        int j = 0;
        bool flagged = false;
        if (valid) {
            b = e / p.N;
            s = ORDERED ? b * p.N + p.row_inv[b * p.row_stride + e - b * p.N] : e;  // the search's position of this point
            const u64 key = p.keys_a[s];
            dmin = __uint_as_float((unsigned)(key >> 32));
            const float* a = p.src + e * 3;
            ax = a[0]; ay = a[1]; az = a[2];
            flagged = ORDERED && p.tie_a[s] == (unsigned)(key >> 32);
            if (!flagged) {
                j = rescan_chunk32(p.tgt_packed + b * (int64_t)p.m_pad * 3, (unsigned)(key & 0xffffffffu), ax, ay, az, dmin);
                if (j >= p.M) j = 0;
                if (ORDERED) j = p.tgt_order[b * p.M + j];
            }
        }
        if (ORDERED) resolve_flagged(flagged, p.tgt, p.M, ax, ay, az, dmin, b, j, p.ties);
        if (!valid) continue;
        const long long* ac = p.acc + e * 3;
        const long long c0 = ac[0], c1 = ac[1], c2 = ac[2];
        const float* t = p.tgt + (b * p.M + j) * 3;
        p.g_src[e * 3 + 0] = g2 * (ax - t[0]) + (float)c0 * inv;
        p.g_src[e * 3 + 1] = g2 * (ay - t[1]) + (float)c1 * inv;
        p.g_src[e * 3 + 2] = g2 * (az - t[2]) + (float)c2 * inv;
        local += (double)dmin;
        if (p.d_fwd) p.d_fwd[e] = dmin;
        if (p.i_fwd) p.i_fwd[e] = j;
        if (p.nn_rows) p.nn_rows[e] = j;
    }
    const double s = block_sum(local, sh);
    if (threadIdx.x == 0) {
        p.partials[col_blocks + blockIdx.x] = s;
        __threadfence();
        last = atomicAdd(p.ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last) {
        // every partial (the column pass finished before this launch started), combined in a FIXED association:
        // thread k adds partials k, k + 256, ... in index order, then a fixed tree over the 256 threads
        __shared__ double tree[kEnergyThreads];
        __threadfence();
        const volatile double* v = p.partials;
        const int n = col_blocks + (int)gridDim.x;
        double tot = 0.0;
        for (int k = threadIdx.x; k < n; k += kEnergyThreads) tot += v[k];
        tree[threadIdx.x] = tot;
        __syncthreads();
        for (int st = kEnergyThreads / 2; st > 0; st >>= 1) {
            if ((int)threadIdx.x < st) tree[threadIdx.x] += tree[threadIdx.x + st];
            __syncthreads();
        }
        if (threadIdx.x == 0) *p.loss = tree[0];
    }
}

// Workspace words behind EnergyParams: acc [B,N,3] int64 | ticket | col_bound must be ZERO before the search runs
// (capi.cu clears them with one memset); partials need no initialisation.
int energy_max_blocks() { return 148 * 16; }

int launch_energy_bwd(const EnergyParams& p, cudaStream_t stream) {
    if (p.B <= 0) return kOk;
    const int64_t rows = (int64_t)p.B * p.N, cols = (int64_t)p.B * p.M;
    if (rows <= 0 || cols <= 0) {                      // a side is empty: no pairs, zero loss and gradient
        if (rows > 0 && cudaMemsetAsync(p.g_src, 0, sizeof(float) * (size_t)rows * 3, stream) != cudaSuccess) return kErrLaunch;
        if (cudaMemsetAsync(p.loss, 0, sizeof(double), stream) != cudaSuccess) return kErrLaunch;
        return kOk;
    }
    if (!p.acc || !p.col_bound || !p.partials || !p.ticket || !p.src_xq || !p.src_perm || p.col_chunk_pts != kSortedChunk ||
        p.row_chunk_pts != kChunk)
        return kErrInvalidArg;
    const int col_blocks = (int)std::min<int64_t>(ceil_div(cols, kEnergyThreads), energy_max_blocks());
    const int row_blocks = (int)std::min<int64_t>(ceil_div(rows, kEnergyThreads), energy_max_blocks());
    if (p.row_order) {
        if (!p.row_inv || !p.tgt_order || !p.tgt_inv || !p.tie_a || !p.tie_b) return kErrInvalidArg;
        energy_cols_kernel<true><<<col_blocks, kEnergyThreads, 0, stream>>>(p);
        REART_CHECK_LAUNCH();
        energy_rows_kernel<true><<<row_blocks, kEnergyThreads, 0, stream>>>(p, col_blocks);
    } else {
        energy_cols_kernel<false><<<col_blocks, kEnergyThreads, 0, stream>>>(p);
        REART_CHECK_LAUNCH();
        energy_rows_kernel<false><<<row_blocks, kEnergyThreads, 0, stream>>>(p, col_blocks);
    }
    REART_CHECK_LAUNCH();
    return kOk;
}

}  // namespace reart
