// cull.cu -- the static bounds the culled search schedule (chamfer_sym.cu, CULL = true) tests against.
//
// The brute-force search evaluates every (skinned point, observed point) pair of a frame.  ANY real point of the other
// cloud bounds a point's minimum from above, and two cheap sources give good ones:
//   * history: an optimisation moves the clouds a little per iteration, so the arg-mins of the PREVIOUS evaluation -- the
//     point's own and those of its neighbours in the caller's point order -- are excellent candidates now
//         ub_i = min over candidates j of d(a_i, b_j)  >=  min_j d(a_i, b_j);
//   * no history: a three-level descent over the other cloud (coarse_upper_bound below), for clouds of >= 8192 points.
// One pass per side turns them into
//   rowbound[b][rc]  = max of ub over the 256 rows of row chunk rc   (one warp of the search owns exactly these rows)
//   colbox[b][cc]    = bounding box of the 32 targets of chunk cc, and the max of ub over them,
// and the search skips a (row chunk, target chunk) pair whose box-to-box squared gap -- a lower bound of every computed
// pair distance in it -- is STRICTLY above both bounds: such a pair can hold neither a minimum nor a tie.  Without seeds
// (nn = -1) and below 8192 points the bounds are infinite and the search is the brute force.  The distances here use the
// very arithmetic of the search (sqdist_scalar), so the bounds bound the COMPUTED minima and the culled keys are
// bit-identical.  How much is skipped depends on how compact the chunks are: the ordered entries of capi.cu run the search
// on copies in a compact order (fixed, or per frame on the posed cloud), and the seeds, kept by caller index, are
// translated through it here; any order is correct.
#include "common.cuh"
#include "kernels.h"
#include <algorithm>

namespace reart {

constexpr int kCullRowChunk = 256;
constexpr int kCullSeeds = 4;                                 // neighbours on each side whose seeds are also tried
constexpr int kCoarse = 256;                                  // points per level-A representative of the coarse descent

// History-free upper bound of min_j d(q, pts_j): a three-level descent over the caller's point order (spatially coherent
// when the caller sorted the cloud): (A) one representative per 256 points, staged in shared memory by the block -> the two
// best; (B) the 8 representatives (one per 32 points) of the best (and a close runner-up) -> the best 32-point chunk; (C)
// every point of it.
// Every candidate is a real point of the cloud and the distance is the search's own arithmetic, so whatever the descent
// finds bounds the computed minimum from above; how tight it is only decides how much is culled.  ~ n/256 + 8..16 + 32
// evaluations per query instead of n.
__device__ __forceinline__ float coarse_upper_bound(const float* __restrict__ pts, int n, const float* __restrict__ s_rep,
                                                    int nrep, float qx, float qy, float qz) {
    float a0 = INFINITY, a1 = INFINITY;
    int r0 = 0, r1 = 0;
    for (int r = 0; r < nrep; ++r) {
        const float d = sqdist_scalar(qx, qy, qz, s_rep[3 * r], s_rep[3 * r + 1], s_rep[3 * r + 2]);
        if (d < a0) { a1 = a0; r1 = r0; a0 = d; r0 = r; }
        else if (d < a1) { a1 = d; r1 = r; }
    }
    float ub = a0;                                             // the representatives are real points
    // (B) the 8 chunk representatives of the best 256-point group (and of the runner-up only when it is close: within 2x
    // in distance), (C) every point of the best chunk -- the global-memory part of the descent, ~20 sectors per query
    float b0 = INFINITY;
    int c0 = -1;
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
        const int r = h ? r1 : r0;
        if (h && (r1 == r0 || !(a1 < 4.0f * a0))) break;
        for (int k = 0; k < kCoarse / kChunk; ++k) {
            const int c = r * (kCoarse / kChunk) + k;
            if (c * kChunk >= n) break;
            const int j = min(c * kChunk + kChunk / 2, n - 1);
            const float* t = pts + (int64_t)j * 3;
            const float d = sqdist_scalar(qx, qy, qz, t[0], t[1], t[2]);
            if (d < b0) { b0 = d; c0 = c; }
        }
    }
    ub = fminf(ub, b0);
    if (c0 >= 0) {
        const int j0 = c0 * kChunk, j1 = min(j0 + kChunk, n);
        if (j1 - j0 == kChunk && ((reinterpret_cast<uintptr_t>(pts + (int64_t)j0 * 3) & 15) == 0)) {
            // a full chunk is 384 contiguous bytes: 24 vector loads instead of 96 scalar ones, four points per three float4
            const float4* v = reinterpret_cast<const float4*>(pts + (int64_t)j0 * 3);
#pragma unroll 2
            for (int g = 0; g < kChunk / 4; ++g) {
                const float4 A = __ldg(v + 3 * g), B = __ldg(v + 3 * g + 1), C = __ldg(v + 3 * g + 2);
                ub = fminf(ub, sqdist_scalar(qx, qy, qz, A.x, A.y, A.z));
                ub = fminf(ub, sqdist_scalar(qx, qy, qz, A.w, B.x, B.y));
                ub = fminf(ub, sqdist_scalar(qx, qy, qz, B.z, B.w, C.x));
                ub = fminf(ub, sqdist_scalar(qx, qy, qz, C.y, C.z, C.w));
            }
        } else {
            for (int j = j0; j < j1; ++j) {
                const float* t = pts + (int64_t)j * 3;
                ub = fminf(ub, sqdist_scalar(qx, qy, qz, t[0], t[1], t[2]));
            }
        }
    }
    return ub;                                                 // NaN coordinates give NaN -> the callers turn that into +inf
}

// stage the level-A representatives of one cloud [n,3]: point min(256 r + 128, n - 1) for r < ceil(n / 256)
__device__ __forceinline__ void coarse_stage(const float* __restrict__ pts, int n, float* s_rep, int nrep) {
    for (int e = threadIdx.x; e < nrep * 3; e += blockDim.x) {
        const int r = e / 3, k = e - 3 * r;
        s_rep[e] = pts[(int64_t)min(r * kCoarse + kCoarse / 2, n - 1) * 3 + k];
    }
}

__global__ void __launch_bounds__(kCullRowChunk) cull_row_bounds_kernel(const CullParams p, int row_chunks, int nrep) {
    extern __shared__ float s_rep[];                           // coarse: [nrep][3] representatives of this frame's targets
    __shared__ unsigned s_w[kCullRowChunk / 32];
    const int rc = blockIdx.x, b = blockIdx.y;
    const int i = rc * kCullRowChunk + threadIdx.x;
    if (p.coarse) {
        coarse_stage(p.b + (int64_t)b * p.nb * 3, p.nb, s_rep, nrep);
        __syncthreads();
    }
    unsigned bits = 0u;                                        // distances are >= 0: their bit patterns order like the floats
    if (i < p.na) {
        // candidates: the row's own previous arg-min and those of its neighbours in the caller's point order (spatial
        // neighbours when the caller sorted the cloud, engine.py) -- a point that changed part since the last step has a
        // useless seed of its own, but a neighbour that already belongs to the new part has a good one.  ANY real target
        // bounds the minimum from above, so the smallest of the candidates is still an exact bound.
        float ub = INFINITY;
        const float* a = p.a + ((int64_t)b * p.na + i) * 3;
        const float ax = a[0], ay = a[1], az = a[2];
        if (p.coarse) {
            ub = coarse_upper_bound(p.b + (int64_t)b * p.nb * 3, p.nb, s_rep, nrep, ax, ay, az);
            if (!(ub >= 0.f)) ub = INFINITY;                   // NaN input: no culling
        }
        if (p.nn_rows) {
            // seeds are kept by caller index: the neighbours' caller rows, their seeds translated into the search order
            int jprev = -2;
#pragma unroll
            for (int d = -kCullSeeds; d <= kCullSeeds; ++d) {
                const int in = min(max(i + d, 0), p.na - 1);
                const int cr = p.row_order ? p.row_order[(int64_t)b * p.row_stride + in] : in;
                const int j = p.nn_rows[(int64_t)b * p.na + cr];
                if (j == jprev) continue;                      // neighbours very often share a seed
                jprev = j;
                if (j >= 0 && j < p.nb) {
                    const int js = p.tgt_inv ? p.tgt_inv[(int64_t)b * p.nb + j] : j;
                    const float* t = p.b + ((int64_t)b * p.nb + js) * 3;
                    const float c = sqdist_scalar(ax, ay, az, t[0], t[1], t[2]);
                    if (c < ub) ub = c;                        // NaN never passes: no culling on NaN input
                }
            }
        }
        bits = __float_as_uint(ub);
    }
    bits = __reduce_max_sync(0xffffffffu, bits);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = bits;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned m = 0u;
#pragma unroll
        for (int w = 0; w < kCullRowChunk / 32; ++w) m = max(m, s_w[w]);
        p.rowbound[(int64_t)b * row_chunks + rc] = __uint_as_float(m);
    }
}

// one warp per 32-target chunk
__global__ void __launch_bounds__(256) cull_col_boxes_kernel(const CullParams p, int chunks_total, int nrep) {
    extern __shared__ float s_rep[];                           // coarse: [nrep][3] representatives of this frame's rows
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.y;
    if (p.coarse) {
        coarse_stage(p.a + (int64_t)b * p.na * 3, p.na, s_rep, nrep);
        __syncthreads();
    }
    const int cc = (int)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (cc >= chunks_total) return;
    const int64_t w = (int64_t)b * chunks_total + cc;
    const int j = cc * kChunk + lane;
    float lx = INFINITY, ly = INFINITY, lz = INFINITY, hx = -INFINITY, hy = -INFINITY, hz = -INFINITY;
    unsigned bits = 0u;
    if (j < p.nb) {
        const float* t = p.b + ((int64_t)b * p.nb + j) * 3;
        const float x = t[0], y = t[1], z = t[2];
        lx = hx = x; ly = hy = y; lz = hz = z;
        // candidates: the previous arg-min rows of this target and of its neighbours in the caller's order, and the rows
        // next to the own one (a row that changed part moved away; its neighbours in the canonical order mostly did not)
        float ub = INFINITY;
        if (p.coarse) {
            ub = coarse_upper_bound(p.a + (int64_t)b * p.na * 3, p.na, s_rep, nrep, x, y, z);
            if (!(ub >= 0.f)) ub = INFINITY;
        }
        if (p.nn_cols) {
#pragma unroll
            for (int d = -kCullSeeds; d <= kCullSeeds; ++d) {
                const int jn = min(max(j + d, 0), p.nb - 1);
                const int cj = p.tgt_order ? p.tgt_order[(int64_t)b * p.nb + jn] : jn;
                const int ic = p.nn_cols[(int64_t)b * p.nb + cj];
                if (ic < 0 || ic >= p.na) continue;
                const int i0 = p.row_inv ? p.row_inv[(int64_t)b * p.row_stride + ic] : ic;
#pragma unroll
                for (int e = -1; e <= 1; ++e) {
                    if (d != 0 && e != 0) continue;            // row neighbours only around the target's own seed
                    const int i = min(max(i0 + e, 0), p.na - 1);
                    const float* a = p.a + ((int64_t)b * p.na + i) * 3;
                    const float c = sqdist_scalar(a[0], a[1], a[2], x, y, z);
                    if (c < ub) ub = c;
                }
            }
        }
        bits = __float_as_uint(ub);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lx = fminf(lx, __shfl_xor_sync(0xffffffffu, lx, o)); ly = fminf(ly, __shfl_xor_sync(0xffffffffu, ly, o));
        lz = fminf(lz, __shfl_xor_sync(0xffffffffu, lz, o)); hx = fmaxf(hx, __shfl_xor_sync(0xffffffffu, hx, o));
        hy = fmaxf(hy, __shfl_xor_sync(0xffffffffu, hy, o)); hz = fmaxf(hz, __shfl_xor_sync(0xffffffffu, hz, o));
    }
    bits = __reduce_max_sync(0xffffffffu, bits);
    if (lane == 0) {
        float4* o = reinterpret_cast<float4*>(p.colbox + w * 8);
        o[0] = make_float4(lx, ly, lz, hx);
        o[1] = make_float4(hy, hz, __uint_as_float(bits), 0.f);
    }
}

int launch_cull_bounds(const CullParams& p, cudaStream_t stream) {
    if (p.B <= 0 || p.na <= 0 || p.nb <= 0) return kOk;
    if (p.B > 65535) return kErrUnsupported;
    const int row_chunks = (int)ceil_div(p.na, kCullRowChunk);
    const int chunks_total = p.nb_pad / kChunk;
    dim3 grid((unsigned)row_chunks, (unsigned)p.B);
    const int nrep_b = p.coarse ? (int)ceil_div(p.nb, kCoarse) : 0, nrep_a = p.coarse ? (int)ceil_div(p.na, kCoarse) : 0;
    if ((size_t)std::max(nrep_a, nrep_b) * 12 > 40 * 1024) return kErrUnsupported;      // clouds beyond 873 k points: no coarse bounds
    cull_row_bounds_kernel<<<grid, kCullRowChunk, (size_t)nrep_b * 12, stream>>>(p, row_chunks, nrep_b);
    REART_CHECK_LAUNCH();
    dim3 cgrid((unsigned)ceil_div(chunks_total, 8), (unsigned)p.B);
    cull_col_boxes_kernel<<<cgrid, 256, (size_t)nrep_a * 12, stream>>>(p, chunks_total, nrep_a);
    REART_CHECK_LAUNCH();
    return kOk;
}

}  // namespace reart
