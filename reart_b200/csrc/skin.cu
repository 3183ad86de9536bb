// skin.cu -- soft-assignment skinning of the canonical cloud, forward and backward (HBM-bound).
//
// Replaces the torch composition of networks/model.py:63-69 (BaseModel), :161-165 (KinematicModel)
// and utils/model_utils.py:54-67 (compute_pc_transform):
//     out[t,n,:] = sum_p W[n,p] * (R[t,p] @ cano[n] + tr[t,p])
// without materialising the [T,P,N,3] intermediate the reference builds with bmm (P x the output).
// Exact zeros in W are skipped (gumbel_softmax(hard=True) / one_hot rows have one non-zero, SURVEY Q5/Q7),
// so the common case costs one 3x4 transform per (t,n).
//
// Algorithmic HBM bytes (DESIGN.md): fwd reads 12N + 4NP + 48TP, writes 12TN (+12TN for the packed copy);
// bwd reads 12TN + 12N + 4NP + 48TP, writes 4NP + 48TP.
#include "common.cuh"
#include "kernels.h"
#include <algorithm>

namespace reart {

constexpr int kSkinThreads = 128;
constexpr int kSkinFramesPerBlock = 8;

// grid (ceil(Npad/128), ceil(T/8)); dynamic smem: [8 frames][P][12] transforms
__global__ void __launch_bounds__(kSkinThreads) skin_fwd_kernel(const float* __restrict__ cano,
                                                                const float* __restrict__ W,
                                                                const float* __restrict__ R,
                                                                const float* __restrict__ tr, int T, int N, int P,
                                                                float* __restrict__ out, float* __restrict__ out_packed,
                                                                int n_pad, int fpb) {
    extern __shared__ float sm_tf[];                          // [frames][P][12]: r00..r22, t0..t2
    const int t0 = blockIdx.y * fpb;
    const int nt = min(fpb, T - t0);
    for (int e = threadIdx.x; e < nt * P * 12; e += blockDim.x) {
        const int f = e / (P * 12), rem = e - f * P * 12, p = rem / 12, k = rem - p * 12;
        const int64_t tp = (int64_t)(t0 + f) * P + p;
        sm_tf[e] = (k < 9) ? R[tp * 9 + k] : tr[tp * 3 + (k - 9)];
    }
    __syncthreads();
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= n_pad) return;
    const bool real = n < N;
    float cx = 0.f, cy = 0.f, cz = 0.f;
    if (real) { cx = cano[3 * n]; cy = cano[3 * n + 1]; cz = cano[3 * n + 2]; }
    const float* __restrict__ w = W + (int64_t)(real ? n : 0) * P;
    for (int f = 0; f < nt; ++f) {
        float ax = 0.f, ay = 0.f, az = 0.f;
        if (real) {
            const float* tf = sm_tf + f * P * 12;
            for (int p = 0; p < P; ++p) {
                const float wp = __ldg(w + p);
                if (wp != 0.f) {
                    const float* m = tf + p * 12;
                    // pinned operation order (common.cuh skin_axis): the fused producer of chamfer_sym.cu must give these bits
                    ax = __fmaf_rn(wp, skin_axis(cx, cy, cz, m[0], m[1], m[2], m[9]), ax);
                    ay = __fmaf_rn(wp, skin_axis(cx, cy, cz, m[3], m[4], m[5], m[10]), ay);
                    az = __fmaf_rn(wp, skin_axis(cx, cy, cz, m[6], m[7], m[8], m[11]), az);
                }
            }
            float* o = out + ((int64_t)(t0 + f) * N + n) * 3;
            o[0] = ax; o[1] = ay; o[2] = az;
        } else {
            ax = ay = az = INFINITY;                          // padding of the packed copy
        }
        if (out_packed) {
            float* g = out_packed + (int64_t)(t0 + f) * n_pad * 3 + (int64_t)(n >> 2) * kGroupFloats + (n & 3);
            g[0] = ax; g[4] = ay; g[8] = az;
        }
    }
}

int launch_skin_fwd(const float* cano, const float* W, const float* R, const float* tr, int64_t T, int64_t N, int64_t P,
                    float* out, float* out_packed, cudaStream_t stream) {
    if (T <= 0 || N <= 0) return kOk;
    if (P <= 0 || P > 32) return kErrUnsupported;
    const int64_t n_pad = out_packed ? padded_points(N) : N;
    // frames per block: 8 amortises the W-row reads, but few frames (a GPU's shard under strong scaling) need more CTAs
    int fpb = kSkinFramesPerBlock;
    while (fpb > 1 && ceil_div(n_pad, kSkinThreads) * ceil_div(T, fpb) < 2 * 148) fpb /= 2;
    dim3 grid((unsigned)ceil_div(n_pad, kSkinThreads), (unsigned)ceil_div(T, fpb));
    const size_t smem = (size_t)fpb * P * 12 * sizeof(float);
    skin_fwd_kernel<<<grid, kSkinThreads, smem, stream>>>(cano, W, R, tr, (int)T, (int)N, (int)P, out, out_packed,
                                                          (int)n_pad, fpb);
    REART_CHECK_LAUNCH();
    return kOk;
}

// ----------------------------------------------------------------------------- forward, x-sorted packed copy
// Same skinning, but the packed copy is written with every block of kSortBlock (= one column chunk of the symmetric
// search: the 256 consecutive points one warp owns) SORTED BY X, plus perm[t][k] = original offset of the point now at
// sorted position k and xq[t][block][16] = x at sorted positions 15, 31, ..., 255 (the quantile index the column-side
// index recovery probes first, common.cuh rescan_sorted_chunk_q).  The recovery then looks at the x window
// |b.x - a.x| <= sqrt(dmin) instead of testing all 256 candidates.
// The AoS output keeps the original order -- it is what the search and every consumer read.  With a search order
// (`order`, the ordered pipeline of capi.cu) the blocks are 256 consecutive points OF THAT ORDER, and the same points are
// also written in that order to out_search: the rows of a search over permuted copies.
constexpr int kSortBlock = 256;

__global__ void __launch_bounds__(kSortBlock) skin_fwd_sorted_kernel(const float* __restrict__ cano,
                                                                     const float* __restrict__ W,
                                                                     const float* __restrict__ R,
                                                                     const float* __restrict__ tr, int T, int N, int P,
                                                                     float* __restrict__ out,
                                                                     float* __restrict__ out_packed,
                                                                     unsigned char* __restrict__ perm,
                                                                     float* __restrict__ xq, int n_pad, int fpb,
                                                                     const int32_t* __restrict__ order,
                                                                     float* __restrict__ out_search) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    u64* xchg = reinterpret_cast<u64*>(sm_raw);                               // [256]
    float* sx = reinterpret_cast<float*>(xchg + kSortBlock);                  // [3][256]
    float* sm_tf = sx + 3 * kSortBlock;                                       // [fpb][P][12]
    const int t0 = blockIdx.y * fpb;
    const int nt = min(fpb, T - t0);
    for (int e = threadIdx.x; e < nt * P * 12; e += blockDim.x) {
        const int f = e / (P * 12), rem = e - f * P * 12, p = rem / 12, k = rem - p * 12;
        const int64_t tp = (int64_t)(t0 + f) * P + p;
        sm_tf[e] = (k < 9) ? R[tp * 9 + k] : tr[tp * 3 + (k - 9)];
    }
    __syncthreads();
    const int i = threadIdx.x;
    const int base = blockIdx.x * kSortBlock;
    const int n = base + i;                                                   // position in the sorted copy's order
    const bool real = n < N;
    const int c = (order && real) ? order[n] : n;                             // the caller's point
    float cx = 0.f, cy = 0.f, cz = 0.f;
    if (real) { cx = cano[3 * c]; cy = cano[3 * c + 1]; cz = cano[3 * c + 2]; }
    const float* __restrict__ w = W + (int64_t)(real ? c : 0) * P;
    const int nblk = n_pad / kSortBlock;
    for (int f = 0; f < nt; ++f) {
        float ax = INFINITY, ay = INFINITY, az = INFINITY;                    // padding sorts last
        if (real) {
            ax = ay = az = 0.f;
            const float* tf = sm_tf + f * P * 12;
            for (int p = 0; p < P; ++p) {
                const float wp = __ldg(w + p);
                if (wp != 0.f) {
                    const float* m = tf + p * 12;
                    // pinned operation order (common.cuh skin_axis): the fused producer of chamfer_sym.cu must give these bits
                    ax = __fmaf_rn(wp, skin_axis(cx, cy, cz, m[0], m[1], m[2], m[9]), ax);
                    ay = __fmaf_rn(wp, skin_axis(cx, cy, cz, m[3], m[4], m[5], m[10]), ay);
                    az = __fmaf_rn(wp, skin_axis(cx, cy, cz, m[6], m[7], m[8], m[11]), az);
                }
            }
            float* o = out + ((int64_t)(t0 + f) * N + c) * 3;
            o[0] = ax; o[1] = ay; o[2] = az;
            if (out_search) {
                float* os = out_search + ((int64_t)(t0 + f) * N + n) * 3;
                os[0] = ax; os[1] = ay; os[2] = az;
            }
        }
        sx[i] = ax; sx[kSortBlock + i] = ay; sx[2 * kSortBlock + i] = az;      // visible after the sort's first barrier
        const u64 key = block_bitonic_sort256(((u64)orderable_bits(ax) << 32) | (u64)i, xchg);
        const int src = (int)(key & 0xffu);
        const float sxv = sx[src];
        sorted_block_store(out_packed + (int64_t)(t0 + f) * n_pad * 3, blockIdx.x, i, sxv, sx[kSortBlock + src],
                           sx[2 * kSortBlock + src]);
        perm[(int64_t)(t0 + f) * n_pad + base + i] = (unsigned char)src;
        if ((i & 15) == 15) xq[((int64_t)(t0 + f) * nblk + blockIdx.x) * kQuantiles + (i >> 4)] = sxv;
        __syncthreads();                                                       // sx is rewritten by the next frame
    }
}

// Eight frames per CTA, sorted by WARPS: phase 1, thread = point, skins its point for all 8 frames into shared memory and
// writes the AoS rows; ONE barrier; phase 2, warp f sorts frame f's 256 keys by itself (8 keys per lane, register swaps and
// shuffles, common.cuh warp_bitonic_sort256) and writes the sorted block, perm and the quantile index.  The block-wide
// hybrid sort above needs 12 barriers per frame; this is 2 per 8 frames.  Same keys, same arithmetic: identical output.
constexpr int kSortFrames = 8;

__global__ void __launch_bounds__(kSortBlock) skin_fwd_sorted8_kernel(const float* __restrict__ cano,
                                                                      const float* __restrict__ W,
                                                                      const float* __restrict__ R,
                                                                      const float* __restrict__ tr, int T, int N, int P,
                                                                      float* __restrict__ out,
                                                                      float* __restrict__ out_packed,
                                                                      unsigned char* __restrict__ perm,
                                                                      float* __restrict__ xq, int n_pad,
                                                                      const int32_t* __restrict__ order,
                                                                      float* __restrict__ out_search) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    float* sx = reinterpret_cast<float*>(sm_raw);                             // [8 frames][3][256]
    float* sm_tf = sx + kSortFrames * 3 * kSortBlock;                         // [8][P][12]
    const int t0 = blockIdx.y * kSortFrames;
    const int nt = min(kSortFrames, T - t0);
    for (int e = threadIdx.x; e < nt * P * 12; e += blockDim.x) {
        const int f = e / (P * 12), rem = e - f * P * 12, p = rem / 12, k = rem - p * 12;
        const int64_t tp = (int64_t)(t0 + f) * P + p;
        sm_tf[e] = (k < 9) ? R[tp * 9 + k] : tr[tp * 3 + (k - 9)];
    }
    __syncthreads();
    const int i = threadIdx.x;
    const int base = blockIdx.x * kSortBlock;
    const int n = base + i;                                                   // position in the sorted copy's order
    const bool real = n < N;
    const int c = (order && real) ? order[n] : n;                             // the caller's point
    float cx = 0.f, cy = 0.f, cz = 0.f;
    if (real) { cx = cano[3 * c]; cy = cano[3 * c + 1]; cz = cano[3 * c + 2]; }
    const float* __restrict__ w = W + (int64_t)(real ? c : 0) * P;
    // the weight row is read ONCE: rows with at most two non-zeros (one-hot / straight-through rows have one) are kept in
    // registers for all 8 frames; denser rows re-read it per frame.  Non-zeros are applied in increasing p either way.
    int p0 = 0, p1 = 0, nnz = 0;
    float w0 = 0.f, w1 = 0.f;
    if (real) {
        for (int p = 0; p < P; ++p) {
            const float wp = __ldg(w + p);
            if (wp != 0.f) {
                if (nnz == 0) { p0 = p; w0 = wp; }
                else if (nnz == 1) { p1 = p; w1 = wp; }
                ++nnz;
            }
        }
    }
    for (int f = 0; f < nt; ++f) {
        float ax = INFINITY, ay = INFINITY, az = INFINITY;                    // padding sorts last
        if (real) {
            ax = ay = az = 0.f;
            const float* tf = sm_tf + f * P * 12;
            if (nnz <= 2) {
                if (nnz >= 1) {
                    const float* m = tf + p0 * 12;
                    ax = __fmaf_rn(w0, skin_axis(cx, cy, cz, m[0], m[1], m[2], m[9]), ax);
                    ay = __fmaf_rn(w0, skin_axis(cx, cy, cz, m[3], m[4], m[5], m[10]), ay);
                    az = __fmaf_rn(w0, skin_axis(cx, cy, cz, m[6], m[7], m[8], m[11]), az);
                }
                if (nnz == 2) {
                    const float* m = tf + p1 * 12;
                    ax = __fmaf_rn(w1, skin_axis(cx, cy, cz, m[0], m[1], m[2], m[9]), ax);
                    ay = __fmaf_rn(w1, skin_axis(cx, cy, cz, m[3], m[4], m[5], m[10]), ay);
                    az = __fmaf_rn(w1, skin_axis(cx, cy, cz, m[6], m[7], m[8], m[11]), az);
                }
            } else {
                for (int p = 0; p < P; ++p) {
                    const float wp = __ldg(w + p);
                    if (wp != 0.f) {
                        const float* m = tf + p * 12;
                        ax = __fmaf_rn(wp, skin_axis(cx, cy, cz, m[0], m[1], m[2], m[9]), ax);
                        ay = __fmaf_rn(wp, skin_axis(cx, cy, cz, m[3], m[4], m[5], m[10]), ay);
                        az = __fmaf_rn(wp, skin_axis(cx, cy, cz, m[6], m[7], m[8], m[11]), az);
                    }
                }
            }
            float* o = out + ((int64_t)(t0 + f) * N + c) * 3;
            o[0] = ax; o[1] = ay; o[2] = az;
            if (out_search) {
                float* os = out_search + ((int64_t)(t0 + f) * N + n) * 3;
                os[0] = ax; os[1] = ay; os[2] = az;
            }
        }
        float* s = sx + f * 3 * kSortBlock;
        s[i] = ax; s[kSortBlock + i] = ay; s[2 * kSortBlock + i] = az;
    }
    __syncthreads();
    const int f = threadIdx.x >> 5, lane = threadIdx.x & 31;                  // warp f owns frame t0 + f
    if (f >= nt) return;
    const float* s = sx + f * 3 * kSortBlock;
    u64 key[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int e = lane * 8 + r;
        key[r] = ((u64)orderable_bits(s[e]) << 32) | (u64)e;
    }
    warp_bitonic_sort256(key, lane);
    const int nblk = n_pad / kSortBlock;
    float* sorted_b = out_packed + (int64_t)(t0 + f) * n_pad * 3;
    unsigned long long pm = 0ull;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int src = (int)(key[r] & 0xffu), pos = lane * 8 + r;
        const float sxv = s[src];
        sorted_block_store(sorted_b, blockIdx.x, pos, sxv, s[kSortBlock + src], s[2 * kSortBlock + src]);
        pm |= (unsigned long long)src << (8 * r);
        if (r == 7 && (lane & 1)) xq[((int64_t)(t0 + f) * nblk + blockIdx.x) * kQuantiles + (pos >> 4)] = sxv;
    }
    *reinterpret_cast<unsigned long long*>(perm + (int64_t)(t0 + f) * n_pad + base + lane * 8) = pm;
}

int launch_skin_fwd_sorted(const float* cano, const float* W, const float* R, const float* tr, int64_t T, int64_t N,
                           int64_t P, float* out, float* out_packed, unsigned char* perm, float* xq, int64_t n_pad,
                           cudaStream_t stream, const int32_t* order, float* out_search) {
    if (T <= 0 || N <= 0) return kOk;
    if (P <= 0 || P > 32 || n_pad % kSortBlock != 0 || n_pad < N) return kErrUnsupported;
    int fpb = kSkinFramesPerBlock;
    while (fpb > 1 && (n_pad / kSortBlock) * ceil_div(T, fpb) < 2 * 148) fpb /= 2;
    if (fpb == kSortFrames) {                                   // enough frames to give every warp of a CTA one to sort
        dim3 grid8((unsigned)(n_pad / kSortBlock), (unsigned)ceil_div(T, kSortFrames));
        const size_t smem8 = ((size_t)kSortFrames * 3 * kSortBlock + (size_t)kSortFrames * P * 12) * sizeof(float);
        skin_fwd_sorted8_kernel<<<grid8, kSortBlock, smem8, stream>>>(cano, W, R, tr, (int)T, (int)N, (int)P, out, out_packed,
                                                                      perm, xq, (int)n_pad, order, out_search);
        REART_CHECK_LAUNCH();
        return kOk;
    }
    dim3 grid((unsigned)(n_pad / kSortBlock), (unsigned)ceil_div(T, fpb));
    const size_t smem = (size_t)kSortBlock * (8 + 12) + (size_t)fpb * P * 12 * sizeof(float);
    skin_fwd_sorted_kernel<<<grid, kSortBlock, smem, stream>>>(cano, W, R, tr, (int)T, (int)N, (int)P, out, out_packed,
                                                               perm, xq, (int)n_pad, fpb, order, out_search);
    REART_CHECK_LAUNCH();
    return kOk;
}

// ----------------------------------------------------------------------------- backward
// g [T,N,3] -> gW [N,P], gR [T,P,9], gtr [T,P,3]
//   gW[n,p]  = sum_t g[t,n] . (R[t,p] c_n + tr[t,p])                (dense in p: straight-through grads)
//   gR[t,p]  = sum_n W[n,p] g[t,n] c_n^T ;  gtr[t,p] = sum_n W[n,p] g[t,n]
// ONE pass over g (round 1 read it twice, 26.7 MB of DRAM reads for 13.8 MB of gradients) and NO atomics -- every sum
// has a fixed association, so the result is bit-identical from run to run:
//   skin_bwd_fused_kernel   a CTA owns kBwdPoints points and walks the frames in tiles of kBwdFrames; the tile of g is
//                           staged in shared memory (the next tile's loads are already in flight in registers);
//                           gW: thread = (point, frame half), P accumulators in registers over all tiles;
//                           pose: thread = (column (t,k) of G[n,(t,k)] = g (x) [c,1], point half), P accumulators, the
//                           block's W rows broadcast from shared memory -- the skinny GEMM W^T G; the two halves are
//                           added in a fixed order and written to partials[chunk][t][k][p];
//   skin_bwd_reduce_kernel  sums the per-chunk partials in chunk order (8 fixed slices, then a fixed combine).
constexpr int kBwdFrames = 8;
constexpr int kBwdPoints = 128;
constexpr int kBwdThreads = 256;
constexpr int kBwdCols = kBwdFrames * 12;                    // 96 pose columns per tile

template <int PMAX>
__global__ void __launch_bounds__(kBwdThreads) skin_bwd_fused_kernel(const float* __restrict__ cano,
                                                                     const float* __restrict__ W,
                                                                     const float* __restrict__ R,
                                                                     const float* __restrict__ tr,
                                                                     const float* __restrict__ g, int T, int N, int P,
                                                                     float* __restrict__ gW,
                                                                     float* __restrict__ partials, int tiles_per_group) {
    extern __shared__ __align__(16) float sm_dyn[];
    float* sW = sm_dyn;                                        // [kBwdPoints][PMAX]
    float* sC = sW + kBwdPoints * PMAX;                        // [kBwdPoints][3] (+ pad to a multiple of 4 floats)
    float* sG = sC + kBwdPoints * 3;                           // [kBwdFrames][kBwdPoints * 3]
    float* sTF = sG + kBwdFrames * kBwdPoints * 3;             // [kBwdFrames][P][12]
    float* sRed = sTF + kBwdFrames * PMAX * 12;                // [kBwdCols][PMAX + 1]  /  [kBwdPoints][PMAX + 1]
    const int tid = threadIdx.x;
    const int n0 = blockIdx.x * kBwdPoints;
    const int cnt = min(kBwdPoints, N - n0);

    for (int e = tid; e < kBwdPoints * PMAX; e += kBwdThreads) {
        const int i = e / PMAX, p = e - i * PMAX;
        sW[e] = (i < cnt && p < P) ? W[(int64_t)(n0 + i) * P + p] : 0.f;
    }
    for (int e = tid; e < kBwdPoints * 3; e += kBwdThreads) sC[e] = e < cnt * 3 ? cano[(int64_t)n0 * 3 + e] : 0.f;

    // register prefetch of a g tile: kBwdFrames x (kBwdPoints*3 = 384) floats = 3072 floats = 12 per thread
    constexpr int kPer = kBwdFrames * kBwdPoints * 3 / kBwdThreads;             // 12
    float pre[kPer];
    auto prefetch = [&](int t0) {
#pragma unroll
        for (int q = 0; q < kPer; ++q) {
            const int e = q * kBwdThreads + tid;                                 // consecutive threads -> consecutive floats
            const int f = e / (kBwdPoints * 3), r = e - f * (kBwdPoints * 3);
            const bool ok = (t0 + f) < T && r < cnt * 3;
            pre[q] = ok ? __ldg(g + ((int64_t)(t0 + f) * N + n0) * 3 + r) : 0.f;
        }
    };
    const int ntiles_all = (T + kBwdFrames - 1) / kBwdFrames;
    const int tile_lo = blockIdx.y * tiles_per_group, tile_hi = min(tile_lo + tiles_per_group, ntiles_all);
    prefetch(tile_lo * kBwdFrames);

    // gW role: thread = (point pl, frame half fh)
    const int pl = tid % kBwdPoints, fh = tid / kBwdPoints;
    float accW[PMAX];
#pragma unroll
    for (int p = 0; p < PMAX; ++p) accW[p] = 0.f;
    // pose role: thread = (column col of the tile, point half ph), 192 of the 256 threads
    const int col = tid % kBwdCols, ph = tid / kBwdCols;
    const bool pose_thread = tid < 2 * kBwdCols;
    const int cf = col / 12, ck = col - cf * 12;
    const int kk = ck < 9 ? ck / 3 : ck - 9;                  // component of g
    const int cl = ck < 9 ? ck % 3 : -1;                      // component of c (or the constant 1)

    for (int tile = tile_lo; tile < tile_hi; ++tile) {
        const int t0 = tile * kBwdFrames;
        const int nt = min(kBwdFrames, T - t0);
        __syncthreads();                                       // previous tile fully consumed (also orders sW/sC fills)
#pragma unroll
        for (int q = 0; q < kPer; ++q) sG[q * kBwdThreads + tid] = pre[q];
        for (int e = tid; e < nt * P * 12; e += kBwdThreads) {
            const int f = e / (P * 12), rem = e - f * P * 12, p = rem / 12, k = rem - p * 12;
            const int64_t tp = (int64_t)(t0 + f) * P + p;
            sTF[(f * PMAX + p) * 12 + k] = (k < 9) ? R[tp * 9 + k] : tr[tp * 3 + (k - 9)];
        }
        __syncthreads();
        if (tile + 1 < tile_hi) prefetch(t0 + kBwdFrames);     // next tile's loads fly during this tile's math

        // ---- gW: frames fh*4 .. fh*4+3 of the tile
        {
            const float cx = sC[3 * pl], cy = sC[3 * pl + 1], cz = sC[3 * pl + 2];
#pragma unroll
            for (int ff = 0; ff < kBwdFrames / 2; ++ff) {
                const int f = fh * (kBwdFrames / 2) + ff;
                if (f < nt) {
                    const float* gg = sG + f * (kBwdPoints * 3) + 3 * pl;
                    const float gx = gg[0], gy = gg[1], gz = gg[2];
                    const float* tf = sTF + f * PMAX * 12;
#pragma unroll
                    for (int p = 0; p < PMAX; ++p) {
                        if (p < P) {
                            const float* m = tf + p * 12;
                            const float vx = cx * m[0] + cy * m[1] + cz * m[2] + m[9];
                            const float vy = cx * m[3] + cy * m[4] + cz * m[5] + m[10];
                            const float vz = cx * m[6] + cy * m[7] + cz * m[8] + m[11];
                            accW[p] += gx * vx + gy * vy + gz * vz;
                        }
                    }
                }
            }
        }
        // ---- pose: column (cf, ck) over the points of half ph
        float accP[PMAX];
#pragma unroll
        for (int p = 0; p < PMAX; ++p) accP[p] = 0.f;
        if (pose_thread && cf < nt) {
            const float* gcol = sG + cf * (kBwdPoints * 3) + kk;
            const int i0 = ph * (kBwdPoints / 2);
            for (int ii = 0; ii < kBwdPoints / 2; ++ii) {
                const int i = i0 + ii;
                float v = gcol[3 * i];
                if (cl >= 0) v *= sC[3 * i + cl];
                const float4* w4 = reinterpret_cast<const float4*>(sW + i * PMAX);
#pragma unroll
                for (int q = 0; q < PMAX / 4; ++q) {
                    const float4 w = w4[q];
                    accP[4 * q] += w.x * v; accP[4 * q + 1] += w.y * v; accP[4 * q + 2] += w.z * v; accP[4 * q + 3] += w.w * v;
                }
            }
        }
        // combine the two point halves in a fixed order (half 0 + half 1) and emit the tile's partial
        if (pose_thread && ph == 1) {
#pragma unroll
            for (int p = 0; p < PMAX; ++p) sRed[col * (PMAX + 1) + p] = accP[p];
        }
        __syncthreads();
        if (pose_thread && ph == 0 && cf < nt) {
            float* o = partials + (((int64_t)blockIdx.x * T + (t0 + cf)) * 12 + ck) * P;
#pragma unroll
            for (int p = 0; p < PMAX; ++p)
                if (p < P) o[p] = accP[p] + sRed[col * (PMAX + 1) + p];
        }
    }
    // ---- gW: frame half 0 + frame half 1 (fixed order)
    __syncthreads();
    if (fh == 1) {
#pragma unroll
        for (int p = 0; p < PMAX; ++p) sRed[pl * (PMAX + 1) + p] = accW[p];
    }
    __syncthreads();
    if (fh == 0 && pl < cnt) {
        // one frame group: the final gW; several: this group's slice of gWpart [groups][N][P] (summed by the reduce kernel)
        float* o = gW + ((int64_t)blockIdx.y * N + (n0 + pl)) * P;
#pragma unroll
        for (int p = 0; p < PMAX; ++p)
            if (p < P) o[p] = accW[p] + sRed[pl * (PMAX + 1) + p];
    }
}

// partials [chunks][T*12][P] -> gR [T,P,9], gtr [T,P,3].  Block = 32 outputs x 8 chunk slices; slice s adds chunks
// s, s+8, ... in order, then the 8 slices are added in order: a fixed association for every output.
constexpr int kRedSlices = 8;
__global__ void __launch_bounds__(32 * kRedSlices) skin_bwd_reduce_kernel(const float* __restrict__ partials, int chunks,
                                                                          int T, int P, float* __restrict__ gR,
                                                                          float* __restrict__ gtr, int pose_blocks,
                                                                          const float* __restrict__ gWpart, int groups,
                                                                          int64_t NP, float* __restrict__ gW) {
    __shared__ float red[kRedSlices][33];
    if ((int)blockIdx.x >= pose_blocks) {                       // trailing blocks: gW = sum over frame groups, in group order
        const int64_t e = ((int64_t)blockIdx.x - pose_blocks) * blockDim.x + threadIdx.x;
        if (e < NP) {
            float v = gWpart[e];
            for (int q = 1; q < groups; ++q) v += gWpart[(int64_t)q * NP + e];
            gW[e] = v;
        }
        return;
    }
    const int lane = threadIdx.x & 31, s = threadIdx.x >> 5;
    const int64_t outs = (int64_t)T * 12 * P;
    const int64_t o = (int64_t)blockIdx.x * 32 + lane;
    float acc = 0.f;
    if (o < outs)
        for (int c = s; c < chunks; c += kRedSlices) acc += __ldg(partials + (int64_t)c * outs + o);
    red[s][lane] = acc;
    __syncthreads();
    if (s == 0 && o < outs) {
        float v = red[0][lane];
#pragma unroll
        for (int q = 1; q < kRedSlices; ++q) v += red[q][lane];
        const int p = (int)(o % P);
        const int64_t tk = o / P;
        const int k = (int)(tk % 12);
        const int64_t t = tk / 12;
        if (k < 9) gR[(t * P + p) * 9 + k] = v;
        else gtr[(t * P + p) * 3 + (k - 9)] = v;
    }
}

// frame groups: enough CTAs to fill the machine when the cloud alone gives too few 128-point chunks
static int skin_bwd_groups(int64_t T, int64_t N) {
    const int64_t chunks = ceil_div(N, kBwdPoints), ntiles = ceil_div(T, kBwdFrames);
    int64_t groups = 1;
    while (chunks * groups < 3 * 148 && groups * 2 <= ntiles) groups *= 2;
    return (int)groups;
}

int64_t skin_bwd_workspace_floats(int64_t T, int64_t N, int64_t P) {
    if (T <= 0 || N <= 0 || P <= 0) return 0;
    const int64_t groups = skin_bwd_groups(T, N);
    return ceil_div(N, kBwdPoints) * T * 12 * P + (groups > 1 ? groups * N * P : 0);
}

template <int PMAX>
static int launch_skin_bwd_p(const float* cano, const float* W, const float* R, const float* tr, const float* g,
                             int64_t T, int64_t N, int64_t P, float* gW, float* gR, float* gtr, float* partials,
                             cudaStream_t stream) {
    const int chunks = (int)ceil_div(N, kBwdPoints);
    const int groups = skin_bwd_groups(T, N);
    const int tiles_per_group = (int)ceil_div(ceil_div(T, kBwdFrames), groups);
    float* gWpart = groups > 1 ? partials + (int64_t)chunks * T * 12 * P : gW;
    const size_t smem = ((size_t)kBwdPoints * PMAX + kBwdPoints * 3 + (size_t)kBwdFrames * kBwdPoints * 3 +
                         (size_t)kBwdFrames * PMAX * 12 + (size_t)kBwdPoints * (PMAX + 1)) * sizeof(float);
    static bool attr_done[64] = {};
    int devid = 0;
    cudaGetDevice(&devid);
    if (smem > 48 * 1024 && (devid < 0 || devid >= 64 || !attr_done[devid])) {
        if (cudaFuncSetAttribute(skin_bwd_fused_kernel<PMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return kErrUnsupported;
        if (devid >= 0 && devid < 64) attr_done[devid] = true;
    }
    dim3 grid((unsigned)chunks, (unsigned)groups);
    skin_bwd_fused_kernel<PMAX><<<grid, kBwdThreads, smem, stream>>>(cano, W, R, tr, g, (int)T, (int)N, (int)P, gWpart,
                                                                     partials, tiles_per_group);
    REART_CHECK_LAUNCH();
    const int64_t outs = T * 12 * P;
    const int pose_blocks = (int)ceil_div(outs, 32);
    const int gw_blocks = groups > 1 ? (int)ceil_div(N * P, 32 * kRedSlices) : 0;
    skin_bwd_reduce_kernel<<<(unsigned)(pose_blocks + gw_blocks), 32 * kRedSlices, 0, stream>>>(
        partials, chunks, (int)T, (int)P, gR, gtr, pose_blocks, gWpart, groups, N * P, gW);
    REART_CHECK_LAUNCH();
    return kOk;
}

int launch_skin_bwd(const float* cano, const float* W, const float* R, const float* tr, const float* g, int64_t T,
                    int64_t N, int64_t P, float* gW, float* gR, float* gtr, float* partials, cudaStream_t stream) {
    if (P <= 0 || P > 32) return kErrUnsupported;
    if (N <= 0 || T <= 0) {                                      // an empty side: all gradients are zero
        if (T * P > 0) {
            if (cudaMemsetAsync(gR, 0, sizeof(float) * (size_t)(T * P * 9), stream) != cudaSuccess) return kErrLaunch;
            if (cudaMemsetAsync(gtr, 0, sizeof(float) * (size_t)(T * P * 3), stream) != cudaSuccess) return kErrLaunch;
        }
        if (N * P > 0 && cudaMemsetAsync(gW, 0, sizeof(float) * (size_t)(N * P), stream) != cudaSuccess) return kErrLaunch;
        return kOk;
    }
    if (!partials) return kErrWorkspace;
    if (P <= 8) return launch_skin_bwd_p<8>(cano, W, R, tr, g, T, N, P, gW, gR, gtr, partials, stream);
    if (P <= 16) return launch_skin_bwd_p<16>(cano, W, R, tr, g, T, N, P, gW, gR, gtr, partials, stream);
    return launch_skin_bwd_p<32>(cano, W, R, tr, g, T, N, P, gW, gR, gtr, partials, stream);
}

}  // namespace reart
