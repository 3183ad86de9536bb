// order.cu -- the per-frame row order of the culled search on the POSED cloud (reart_skinned_chamfer_fwd_bwd_posed).
//
// How much the culled search skips depends on how compact its 256-row blocks are.  One k-d order of the canonical cloud
// stops being compact once the parts move apart: under gumbel sampling a canonical leaf is scattered over up to P
// differently moved places of every frame.  So every step, after skinning, each frame's rows are grouped again on the
// skinned cloud itself, by a sort-tile-recursive (STR) order on quantised coordinates:
//   * the frame's axes by decreasing bounding-box extent (equal extents: lower axis first);
//   * level 1: rows ordered by (q1, caller index), q1 = the coordinate along the first axis quantised to 4096 cells of
//     the frame's extent, and cut into slabs of 2048 consecutive rows; level 2: rows ordered by (slab, q2, caller index),
//     q2 along the second axis in 512 cells, cut into pieces of 512; level 3: (piece, q3, caller index), 128 cells along
//     the third axis, cut into leaves of 256 (8 x 4 x 2 leaves at 16 384 points; only the last leaf of a frame is short);
//   * every leaf in ascending caller index -- the tie rule of the ordered search needs leaves in caller order
//     (DESIGN.md section 4.4); the culling only needs leaf membership.
// q = min(cells - 1, trunc((x - lo) * (cells / extent))) in float32 round-to-nearest (0 for a zero or non-finite extent):
// the order is deterministic and scripts / tests reproduce it exactly in numpy.
//
// One CTA per frame.  A level is a counting sort in shared memory: a histogram over the 4096 (segment, cell) buckets, a
// scan, a scatter, then every bucket's few rows put in caller-index order (insertion sort by the bucket's owner thread).
// The quantised keys are what makes this O(N) per level instead of a comparison sort's O(N log^2 N) shared-memory passes.
// The same kernel writes everything the search needs in that order: the order and its inverse, the AoS rows in search
// order, and the x-sorted 256-row blocks with perm / xq (as skin_fwd_sorted8_kernel writes them for a fixed order).
#include "common.cuh"
#include "kernels.h"

namespace reart {

constexpr int kOrderThreads = 1024;
constexpr int kOrderBuckets = 4096;
constexpr int kOrderMaxRows = 16384;
// per level: rows per segment (slab, piece, leaf) and cells per segment (segments <= 1, 8, 32: at most 4096 buckets)
__host__ __device__ constexpr int order_size(int lv) { return lv == 0 ? 2048 : lv == 1 ? 512 : 256; }
__host__ __device__ constexpr int order_cells(int lv) { return lv == 0 ? 4096 : lv == 1 ? 512 : 128; }

__device__ __forceinline__ unsigned order_cell(float x, float lo, float scale, int cells) {
    const float v = __fmul_rn(__fsub_rn(x, lo), scale);
    if (!(v > 0.f)) return 0u;                                // also NaN
    return min((unsigned)(cells - 1), __float2uint_rz(v));
}

// shared memory: slot [N] u32 (rows in the current order) | cnt [4096] u32 | start [4096] u32 | seg [N] u8
__global__ void __launch_bounds__(kOrderThreads) posed_order_kernel(const float* __restrict__ skinned, int N, int n_pad,
                                                                     int32_t* __restrict__ row_order,
                                                                     int32_t* __restrict__ row_inv,
                                                                     float* __restrict__ out_search,
                                                                     float* __restrict__ out_packed,
                                                                     unsigned char* __restrict__ perm,
                                                                     float* __restrict__ xq) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    unsigned* slot = reinterpret_cast<unsigned*>(sm_raw);
    unsigned* cnt = slot + kOrderMaxRows;
    unsigned* start = cnt + kOrderBuckets;
    unsigned char* seg = reinterpret_cast<unsigned char*>(start + kOrderBuckets);
    __shared__ float s_ext[kOrderThreads / 32][6];
    __shared__ float s_lo[3], s_scale[3];
    __shared__ int s_axis[3];
    __shared__ unsigned s_wsum[kOrderThreads / 32];
    const int t = blockIdx.x;
    const float* __restrict__ pts = skinned + (int64_t)t * N * 3;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // bounding box of the frame
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int k = threadIdx.x; k < N; k += blockDim.x) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = __ldg(pts + (int64_t)k * 3 + a);
            lo[a] = fminf(lo[a], v); hi[a] = fmaxf(hi[a], v);
        }
        seg[k] = 0;
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        if (lane == 0) { s_ext[warp][a] = lo[a]; s_ext[warp][3 + a] = hi[a]; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float l[3], ext[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            float h = s_ext[0][3 + a];
            l[a] = s_ext[0][a];
            for (int w = 1; w < kOrderThreads / 32; ++w) { l[a] = fminf(l[a], s_ext[w][a]); h = fmaxf(h, s_ext[w][3 + a]); }
            ext[a] = __fsub_rn(h, l[a]);
        }
        int ax[3] = {0, 1, 2};                                 // decreasing extent, lower axis first among equal ones
        for (int u = 0; u < 2; ++u)
            for (int v = 0; v < 2 - u; ++v)
                if (ext[ax[v + 1]] > ext[ax[v]]) { const int s = ax[v]; ax[v] = ax[v + 1]; ax[v + 1] = s; }
#pragma unroll
        for (int lv = 0; lv < 3; ++lv) {
            const float e = ext[ax[lv]];
            s_axis[lv] = ax[lv];
            s_lo[lv] = l[ax[lv]];
            s_scale[lv] = (e > 0.f && e < INFINITY) ? __fdiv_rn((float)order_cells(lv), e) : 0.f;
        }
    }
    __syncthreads();
    for (int lv = 0; lv < 3; ++lv) {
        const int axis = s_axis[lv], cells = order_cells(lv);
        const float l = s_lo[lv], scale = s_scale[lv];
        for (int b = threadIdx.x; b < kOrderBuckets; b += blockDim.x) cnt[b] = 0u;
        __syncthreads();
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            const unsigned bkt = (unsigned)seg[i] * cells + order_cell(__ldg(pts + (int64_t)i * 3 + axis), l, scale, cells);
            atomicAdd(cnt + bkt, 1u);
        }
        __syncthreads();
        // exclusive scan of the 4096 counts: 4 consecutive buckets per thread, then a block scan of the thread sums
        unsigned c[4], sum = 0u;
#pragma unroll
        for (int r = 0; r < 4; ++r) { c[r] = cnt[threadIdx.x * 4 + r]; sum += c[r]; }
        unsigned inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        if (lane == 31) s_wsum[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            unsigned w = s_wsum[lane], wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned v = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += v;
            }
            s_wsum[lane] = wi - w;
        }
        __syncthreads();
        unsigned run = s_wsum[warp] + inc - sum;
#pragma unroll
        for (int r = 0; r < 4; ++r) { start[threadIdx.x * 4 + r] = run; cnt[threadIdx.x * 4 + r] = run; run += c[r]; }
        __syncthreads();
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            const unsigned bkt = (unsigned)seg[i] * cells + order_cell(__ldg(pts + (int64_t)i * 3 + axis), l, scale, cells);
            slot[atomicAdd(cnt + bkt, 1u)] = (unsigned)i;
        }
        __syncthreads();
        // every bucket in caller-index order (cnt[b] is now the bucket's end)
        for (int b = threadIdx.x; b < kOrderBuckets; b += blockDim.x) {
            const unsigned s0 = start[b], s1 = cnt[b];
            for (unsigned u = s0 + 1; u < s1; ++u) {
                const unsigned v = slot[u];
                unsigned w = u;
                while (w > s0 && slot[w - 1] > v) { slot[w] = slot[w - 1]; --w; }
                slot[w] = v;
            }
        }
        __syncthreads();
        for (int k = threadIdx.x; k < N; k += blockDim.x) seg[slot[k]] = (unsigned char)(k / order_size(lv));
        __syncthreads();
    }
    // leaves (256 consecutive rows of the level-3 order) in caller-index order: one warp per leaf
    const int nblk = n_pad / kSortedChunk;
    for (int blk = warp; blk < nblk; blk += kOrderThreads / 32) {
        u64 key[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int k = blk * kSortedChunk + lane * 8 + r;
            key[r] = k < N ? (u64)slot[k] : ~0ull;
        }
        warp_bitonic_sort256(key, lane);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int k = blk * kSortedChunk + lane * 8 + r;
            if (k < N) slot[k] = (unsigned)key[r];
        }
    }
    __syncthreads();
    // the order, its inverse and the rows in search order
    for (int k = threadIdx.x; k < N; k += blockDim.x) {
        const int idx = (int)slot[k];
        row_order[(int64_t)t * N + k] = idx;
        row_inv[(int64_t)t * N + idx] = k;
        const float* p = pts + (int64_t)idx * 3;
        float* o = out_search + ((int64_t)t * N + k) * 3;
        o[0] = __ldg(p); o[1] = __ldg(p + 1); o[2] = __ldg(p + 2);
    }
    // the x-sorted 256-row blocks of that order: one warp per block (skin_fwd_sorted8_kernel's keys and stores)
    float* sorted_b = out_packed + (int64_t)t * n_pad * 3;
    for (int blk = warp; blk < nblk; blk += kOrderThreads / 32) {
        u64 kx[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int e = lane * 8 + r, k = blk * kSortedChunk + e;
            const float x = k < N ? __ldg(pts + (int64_t)slot[k] * 3) : INFINITY;
            kx[r] = ((u64)orderable_bits(x) << 32) | (u64)e;
        }
        warp_bitonic_sort256(kx, lane);
        unsigned long long pm = 0ull;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int src = (int)(kx[r] & 0xffu), pos = lane * 8 + r, k = blk * kSortedChunk + src;
            float x = INFINITY, y = INFINITY, z = INFINITY;
            if (k < N) {
                const float* p = pts + (int64_t)slot[k] * 3;
                x = __ldg(p); y = __ldg(p + 1); z = __ldg(p + 2);
            }
            sorted_block_store(sorted_b, blk, pos, x, y, z);
            pm |= (unsigned long long)src << (8 * r);
            if (r == 7 && (lane & 1)) xq[((int64_t)t * nblk + blk) * kQuantiles + (pos >> 4)] = x;
        }
        *reinterpret_cast<unsigned long long*>(perm + (int64_t)t * n_pad + blk * kSortedChunk + lane * 8) = pm;
    }
}

int posed_order_max_points() { return kOrderMaxRows; }

int launch_posed_order(const float* skinned, int64_t T, int64_t N, int64_t n_pad, int32_t* row_order, int32_t* row_inv,
                       float* out_search, float* out_packed, unsigned char* perm, float* xq, cudaStream_t stream) {
    if (T <= 0 || N <= 0) return kOk;
    if (N > kOrderMaxRows || T > 0x7fffffff || n_pad % kSortedChunk != 0 || n_pad < N) return kErrUnsupported;
    const size_t smem = (size_t)kOrderMaxRows * 4 + 2 * (size_t)kOrderBuckets * 4 + kOrderMaxRows;
    static bool attr_done[64] = {};
    int devid = -1;
    cudaGetDevice(&devid);
    if (devid < 0 || devid >= 64 || !attr_done[devid]) {
        if (cudaFuncSetAttribute(posed_order_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return kErrUnsupported;
        if (devid >= 0 && devid < 64) attr_done[devid] = true;
    }
    posed_order_kernel<<<(unsigned)T, kOrderThreads, smem, stream>>>(skinned, (int)N, (int)n_pad, row_order, row_inv,
                                                                     out_search, out_packed, perm, xq);
    REART_CHECK_LAUNCH();
    return kOk;
}

}  // namespace reart
