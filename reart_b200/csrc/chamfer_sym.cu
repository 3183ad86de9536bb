// chamfer_sym.cu -- bidirectional K=1 search that evaluates every (a_i, b_j) distance ONCE and
// feeds both directions (row min for a_i over B, column min for b_j over A).
//
// Replaces the two chamferdist._C.knn_points_idx calls of ChamferDistance.forward
// (utils/chamfer.py:78-94).  d(a,b) = fma(dz,dz,fma(dy,dy,dx*dx)) is bit-symmetric in (a,b)
// (dx -> -dx squares to the same value), so one evaluation serves both oracle searches exactly.
//
// Why: measured on B200 the FMA pipe and the issue port are the same resource for this loop
// (packed FADD2/FMUL2/FFMA2 occupy two issue slots each, FMNMX one; profiles/r01_fp32_probes.md),
// so a one-direction sweep costs 6 + 1 slots per pair = at most 57 % of FP32 peak.  Sharing the
// distance costs 6 + 1 (row) + 1 (column) + ~0.1 slots per TWO directed pairs.
//
// Layout: thread (warp w, lane l) keeps R consecutive A points  i = qbase + (32 w + l) R + r  in
// registers; B streams through shared memory exactly as in knn1.cu (TMA bulk ring).  Row side:
// running min + 32-target chunk id (as knn1.cu).  Column side: per target the lane folds its R
// distances (FMNMX), the warp folds lanes with one REDUX.MIN on the bit pattern, lane 0 stores the
// warp's value into a per-warp shared array; after each tile the CTA reduces the 8 warp arrays and
// merges into global keys with 64-bit atomicMin (dist_bits<<32 | column-chunk), where a column
// chunk is the 32*R consecutive A points owned by one warp.  Indices are recovered by the
// finalize re-scan (knn1.cu) with chunk sizes 32 (rows) and 32*R (columns).
#include "common.cuh"
#include "kernels.h"
#include <algorithm>

namespace reart {

constexpr int kSymStages = 3;
constexpr int kSymThreads = 256;
constexpr int kSymWarps = kSymThreads / 32;

// R  = A points per thread (registers); S = column sub-chunks per warp: the lane's R distances to a target are
// folded in S groups of R/S, each group goes through its own REDUX, so a column chunk is 32*R/S consecutive A
// points.  In-lane folds + REDUX count R per target for every S, yet larger S measured slower on B200 (more
// predicated stores, a wider per-tile fold, smaller tiles), so S=1 is the production setting; S is also bounded by shared memory
// (2 buffers x 8 warps x S x tile points x 4 B), which is why the tile shrinks as S grows.
template <int R, int S>
struct SymCfg {
    static constexpr int kTileChunks = S <= 2 ? 16 : (S == 4 ? 8 : 4);
    static constexpr int kTilePoints = kTileChunks * kChunk;
    static constexpr int kTileBytes = kTilePoints * 12;
    static constexpr int kColBufs = 2;
    static constexpr int kColBufWords = kSymWarps * S * kTilePoints;
    static constexpr size_t kSmem = (size_t)kSymStages * kTileBytes + (size_t)kColBufs * kColBufWords * 4;
    static constexpr int kColChunkPts = 32 * R / S;
};

// CULL = true adds the exact tile culling of DESIGN.md section 4.4: every 32-target chunk arrives with its bounding box
// and an upper bound of its columns' final minima (cull.cu), every warp knows the box of its 256 rows and an upper bound
// of their final minima; a (warp, chunk) pair whose box-to-box squared gap -- formed with the same subtract / multiply /
// fma sequence as a point distance, hence a lower bound of every computed pair distance -- is STRICTLY larger than both
// bounds cannot contain a minimum or a tie of either side and is skipped.  Keys are bit-identical to the brute force.
constexpr int kBoxFloats = 8;                                  // lo.xyz, hi.xyz, column bound, pad  (32 B per chunk)

// SKIN = true is the fused PRODUCER (the north-star design, SURVEY N1): the A rows are not read from memory, every CTA
// skins its 2048 canonical points itself in the prologue -- one-hot weights in compact form (part, value), the frame's
// P transforms staged in shared memory -- with the pinned arithmetic of skin.cu (common.cuh skin_axis), so the rows are
// bit-identical to what skin_fwd_sorted_kernel writes.  The CTAs of the first target split also emit what the later
// passes read: the AoS skinned cloud, and per warp the x-sorted copy of its 256 rows with perm and the quantile index
// (a warp-level bitonic sort, no barrier).  This removes the skin launch and the re-read of the skinned cloud.
template <int R, int S, bool CULL, bool SKIN>
__global__ void __launch_bounds__(kSymThreads, 2) chamfer_sym_kernel(const SymParams p) {
    using C = SymCfg<R, S>;
    static_assert(!SKIN || (R == 8 && S == 1 && !CULL), "the fused producer is built for the production configuration");
    __shared__ float s_tf[SKIN ? 32 * 12 : 1];                // SKIN: [P][12] transforms of this frame
    constexpr int RS = R / S;                                  // points per lane per sub-chunk
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // [stages][tile bytes] | [2][warps][S][tile points] u32 | CULL: [stages][tile chunks][8] f32 boxes
    unsigned* colmin = reinterpret_cast<unsigned*>(smem_raw + kSymStages * C::kTileBytes);
    float* sbox = reinterpret_cast<float*>(smem_raw + C::kSmem);
    __shared__ __align__(8) uint64_t full_bar[kSymStages];

    int item = blockIdx.x;
    const int qb = item % p.qblocks;
    item /= p.qblocks;
    const int split = item % p.splits;
    const int b = item / p.splits;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int QB = R * kSymThreads;
    const int qbase = qb * QB;
    const float* __restrict__ q = p.a + (int64_t)b * p.na * 3;

    const int chunks_total = p.nb_pad / kChunk;
    const int cps = (chunks_total + p.splits - 1) / p.splits;
    const int chunk0 = split * cps;
    const int nchunks = min(cps, chunks_total - chunk0);
    const int ntiles = (nchunks + C::kTileChunks - 1) / C::kTileChunks;
    const float* __restrict__ tp = p.b_packed + (int64_t)b * p.nb_pad * 3 + (int64_t)chunk0 * kChunk * 3;
    u64* __restrict__ keys_col = p.keys_b + (int64_t)b * p.nb;
    const unsigned colchunk_base = (unsigned)(qbase / C::kColChunkPts);

    unsigned cmax = 0u;                                      // largest finite column minimum this thread merged

    const float* __restrict__ bp = CULL ? p.colbox + ((int64_t)b * chunks_total + chunk0) * kBoxFloats : nullptr;
    auto issue = [&](int k) {
        const int st = k % kSymStages;
        const int nch = min(C::kTileChunks, nchunks - k * C::kTileChunks);
        const uint32_t bytes = (uint32_t)nch * kChunk * 12;
        const uint32_t box_bytes = CULL ? (uint32_t)nch * kBoxFloats * 4 : 0u;
        mbar_expect_tx(&full_bar[st], bytes + box_bytes);
        tma_bulk_g2s(smem_raw + st * C::kTileBytes, tp + (int64_t)k * C::kTilePoints * 3, bytes, &full_bar[st]);
        if (CULL)
            tma_bulk_g2s(sbox + st * C::kTileChunks * kBoxFloats, bp + (int64_t)k * C::kTileChunks * kBoxFloats, box_bytes,
                         &full_bar[st]);
    };
    // the first tiles are requested BEFORE the rows are loaded: the TMA latency of a work item hides behind its own
    // prologue (small shards under strong scaling run items of a single tile, where it was fully exposed)
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kSymStages; ++s) mbar_init(&full_bar[s], 1);
        mbar_fence_init();
        for (int k = 0; k < min(kSymStages, ntiles); ++k) issue(k);
    }


    // register r = s*RS + rr holds A point  qbase + warp*32R + s*(32 RS) + lane*RS + rr
    u64 QX[R], QY[R], QZ[R];
    float best[R], prev[R];
    unsigned bch[R];
    float rlx = INFINITY, rly = INFINITY, rlz = INFINITY, rhx = -INFINITY, rhy = -INFINITY, rhz = -INFINITY;
    if (SKIN) {
        // ---- fused producer: skin this thread's 8 consecutive canonical points
        for (int e = tid; e < p.sk_P * 12; e += kSymThreads) {
            const int pp = e / 12, k = e - pp * 12;
            const int64_t tpi = (int64_t)b * p.sk_P + pp;
            s_tf[e] = k < 9 ? p.sk_R[tpi * 9 + k] : p.sk_tr[tpi * 3 + (k - 9)];
        }
        __syncthreads();
        const int i0 = qbase + warp * 256 + lane * 8;
        float cf[24];
        int2 hot[8];
        if (i0 + 8 <= p.na) {                                  // 96 B of cano and 64 B of (part, value) per lane: vector loads
            const float4* c4 = reinterpret_cast<const float4*>(p.sk_cano + (int64_t)i0 * 3);
            const int4* h4 = reinterpret_cast<const int4*>(p.sk_hot + (int64_t)i0 * 2);
#pragma unroll
            for (int v = 0; v < 6; ++v) { const float4 t = __ldg(c4 + v); cf[4 * v] = t.x; cf[4 * v + 1] = t.y; cf[4 * v + 2] = t.z; cf[4 * v + 3] = t.w; }
#pragma unroll
            for (int v = 0; v < 4; ++v) { const int4 t = __ldg(h4 + v); hot[2 * v] = make_int2(t.x, t.y); hot[2 * v + 1] = make_int2(t.z, t.w); }
        } else {
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int i = min(i0 + r, p.na - 1);
                cf[3 * r] = p.sk_cano[3 * (int64_t)i]; cf[3 * r + 1] = p.sk_cano[3 * (int64_t)i + 1]; cf[3 * r + 2] = p.sk_cano[3 * (int64_t)i + 2];
                hot[r] = make_int2(__float_as_int(p.sk_hot[2 * (int64_t)i]), __float_as_int(p.sk_hot[2 * (int64_t)i + 1]));
            }
        }
        float xr[8], yr[8], zr[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            xr[r] = yr[r] = zr[r] = INFINITY;                  // out-of-range rows never win a column and sort last
            if (i0 + r < p.na) {
                const float* m = s_tf + min(max(hot[r].x, 0), p.sk_P - 1) * 12;
                const float wv = __int_as_float(hot[r].y);
                const float cx = cf[3 * r], cy = cf[3 * r + 1], cz = cf[3 * r + 2];
                // skin.cu: acc = 0; acc = fma(w, R_row . c + t, acc) for the one non-zero weight
                xr[r] = __fmaf_rn(wv, skin_axis(cx, cy, cz, m[0], m[1], m[2], m[9]), 0.f);
                yr[r] = __fmaf_rn(wv, skin_axis(cx, cy, cz, m[3], m[4], m[5], m[10]), 0.f);
                zr[r] = __fmaf_rn(wv, skin_axis(cx, cy, cz, m[6], m[7], m[8], m[11]), 0.f);
            }
            QX[r] = pack2(xr[r], xr[r]); QY[r] = pack2(yr[r], yr[r]); QZ[r] = pack2(zr[r], zr[r]);
            best[r] = INFINITY; prev[r] = INFINITY; bch[r] = 0u;
        }
        const int blk = qbase / 256 + warp;                    // the 256-point block this warp owns
        const int nblk = p.sk_npad / 256;
        if (split == 0 && blk < nblk) {
            // ---- by-products, written once per (frame, row block): AoS cloud, x-sorted block, perm, quantile index
            float* out = p.sk_out + ((int64_t)b * p.na + i0) * 3;
            if (i0 + 8 <= p.na && (p.na & 3) == 0) {
                float4* o4 = reinterpret_cast<float4*>(out);
                o4[0] = make_float4(xr[0], yr[0], zr[0], xr[1]); o4[1] = make_float4(yr[1], zr[1], xr[2], yr[2]);
                o4[2] = make_float4(zr[2], xr[3], yr[3], zr[3]); o4[3] = make_float4(xr[4], yr[4], zr[4], xr[5]);
                o4[4] = make_float4(yr[5], zr[5], xr[6], yr[6]); o4[5] = make_float4(zr[6], xr[7], yr[7], zr[7]);
            } else {
#pragma unroll
                for (int r = 0; r < 8; ++r)
                    if (i0 + r < p.na) { out[3 * r] = xr[r]; out[3 * r + 1] = yr[r]; out[3 * r + 2] = zr[r]; }
            }
            float* stg = reinterpret_cast<float*>(colmin) + warp * 768;      // the column buffers are idle until the main loop
            u64 key[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int e = lane * 8 + r;
                stg[e] = xr[r]; stg[256 + e] = yr[r]; stg[512 + e] = zr[r];
                key[r] = ((u64)orderable_bits(xr[r]) << 32) | (u64)e;
            }
            __syncwarp();
            warp_bitonic_sort256(key, lane);
            float* sorted_b = p.sk_sorted + (int64_t)b * p.sk_npad * 3;
            unsigned long long pm = 0ull;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int src = (int)(key[r] & 0xffu), pos = lane * 8 + r;
                const float sx = stg[src];
                sorted_block_store(sorted_b, blk, pos, sx, stg[256 + src], stg[512 + src]);
                pm |= (unsigned long long)src << (8 * r);
                if (r == 7 && (lane & 1)) p.sk_xq[((int64_t)b * nblk + blk) * kQuantiles + (pos >> 4)] = sx;
            }
            *reinterpret_cast<unsigned long long*>(p.sk_perm + (int64_t)b * p.sk_npad + (int64_t)blk * 256 + lane * 8) = pm;
        }
    } else {
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = qbase + warp * (32 * R) + (r / RS) * (32 * RS) + lane * RS + (r % RS);
        float x = INFINITY, y = INFINITY, z = INFINITY;          // out-of-range rows never win a column
        if (i < p.na) {
            x = q[3 * i]; y = q[3 * i + 1]; z = q[3 * i + 2];
            if (CULL) {
                rlx = fminf(rlx, x); rly = fminf(rly, y); rlz = fminf(rlz, z);
                rhx = fmaxf(rhx, x); rhy = fmaxf(rhy, y); rhz = fmaxf(rhz, z);
            }
        }
        QX[r] = pack2(x, x); QY[r] = pack2(y, y); QZ[r] = pack2(z, z);
        best[r] = INFINITY; prev[r] = INFINITY; bch[r] = 0u;
    }
    }
    float rbound = INFINITY;                                   // upper bound of the final minima of this warp's rows
    unsigned evaluated = 0u;
    if (CULL) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            rlx = fminf(rlx, __shfl_xor_sync(0xffffffffu, rlx, o)); rly = fminf(rly, __shfl_xor_sync(0xffffffffu, rly, o));
            rlz = fminf(rlz, __shfl_xor_sync(0xffffffffu, rlz, o)); rhx = fmaxf(rhx, __shfl_xor_sync(0xffffffffu, rhx, o));
            rhy = fmaxf(rhy, __shfl_xor_sync(0xffffffffu, rhy, o)); rhz = fmaxf(rhz, __shfl_xor_sync(0xffffffffu, rhz, o));
        }
        const int rc = qbase / (32 * R) + warp;                // this warp's 256-row chunk
        if (rc * (32 * R) < p.na) rbound = __ldg(p.rowbound + (int64_t)b * p.row_chunks + rc);
    }

    __syncthreads();                                         // barrier initialisation visible to every waiter

    for (int k = 0; k < ntiles; ++k) {
        const int st = k % kSymStages;
        mbar_wait(&full_bar[st], (uint32_t)((k / kSymStages) & 1));
        const int nch = min(C::kTileChunks, nchunks - k * C::kTileChunks);
        const float4* __restrict__ tile = reinterpret_cast<const float4*>(smem_raw + st * C::kTileBytes);
        unsigned* __restrict__ cbuf = colmin + (k & 1) * C::kColBufWords;
        unsigned* __restrict__ cm_w = cbuf + warp * (S * C::kTilePoints);
        for (int c = 0; c < nch; ++c) {
            if (CULL) {
                const float4 b0 = *reinterpret_cast<const float4*>(sbox + (st * C::kTileChunks + c) * kBoxFloats);
                const float4 b1 = *reinterpret_cast<const float4*>(sbox + (st * C::kTileChunks + c) * kBoxFloats + 4);
                // b0 = (lo.x, lo.y, lo.z, hi.x), b1 = (hi.y, hi.z, column bound, -)
                const float gx = fmaxf(0.f, fmaxf(__fsub_rn(rlx, b0.w), __fsub_rn(b0.x, rhx)));
                const float gy = fmaxf(0.f, fmaxf(__fsub_rn(rly, b1.x), __fsub_rn(b0.y, rhy)));
                const float gz = fmaxf(0.f, fmaxf(__fsub_rn(rlz, b1.y), __fsub_rn(b0.z, rhz)));
                const float lb = __fmaf_rn(gz, gz, __fmaf_rn(gy, gy, __fmul_rn(gx, gx)));
                if (lb > rbound && lb > b1.z) {                // warp-uniform: no minimum and no tie of either side in here
                    if (lane == 0) {
                        const uint4 inf4 = make_uint4(0x7f800000u, 0x7f800000u, 0x7f800000u, 0x7f800000u);
#pragma unroll
                        for (int s = 0; s < S; ++s)
#pragma unroll
                            for (int g = 0; g < kChunk / 4; ++g)
                                *reinterpret_cast<uint4*>(cm_w + s * C::kTilePoints + c * kChunk + 4 * g) = inf4;
                    }
                    continue;
                }
                ++evaluated;
            }
            const float4* __restrict__ cg = tile + c * (kChunk / 4 * 3);
#pragma unroll
            for (int g = 0; g < kChunk / 4; ++g) {
                const float4 X = cg[3 * g], Y = cg[3 * g + 1], Z = cg[3 * g + 2];
                const u64 X01 = pack2(X.x, X.y), X23 = pack2(X.z, X.w);
                const u64 Y01 = pack2(Y.x, Y.y), Y23 = pack2(Y.z, Y.w);
                const u64 Z01 = pack2(Z.x, Z.y), Z23 = pack2(Z.z, Z.w);
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    float c0, c1, c2, c3;
#pragma unroll
                    for (int rr = 0; rr < RS; ++rr) {
                        const int r = s * RS + rr;
                        float a0, a1, a2, a3;
                        unpack2(sqdist_pair(QX[r], QY[r], QZ[r], X01, Y01, Z01), a0, a1);
                        unpack2(sqdist_pair(QX[r], QY[r], QZ[r], X23, Y23, Z23), a2, a3);
                        best[r] = min3(best[r], a0, a1);
                        best[r] = min3(best[r], a2, a3);
                        if (rr == 0) { c0 = a0; c1 = a1; c2 = a2; c3 = a3; }
                        else { c0 = fminf(c0, a0); c1 = fminf(c1, a1); c2 = fminf(c2, a2); c3 = fminf(c3, a3); }
                    }
                    const unsigned m0 = __reduce_min_sync(0xffffffffu, __float_as_uint(c0));
                    const unsigned m1 = __reduce_min_sync(0xffffffffu, __float_as_uint(c1));
                    const unsigned m2 = __reduce_min_sync(0xffffffffu, __float_as_uint(c2));
                    const unsigned m3 = __reduce_min_sync(0xffffffffu, __float_as_uint(c3));
                    if (lane == 0)
                        *reinterpret_cast<uint4*>(cm_w + s * C::kTilePoints + c * kChunk + 4 * g) = make_uint4(m0, m1, m2, m3);
                }
            }
            const unsigned gid = (unsigned)(chunk0 + k * C::kTileChunks + c);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (best[r] < prev[r]) bch[r] = gid;
                prev[r] = best[r];
            }
        }
        __syncthreads();                                   // tile consumed, per-warp column minima complete
        if (tid == 0 && k + kSymStages < ntiles) issue(k + kSymStages);
        // fold the warps x S column arrays of this tile and merge into the global column keys; (warp, s) in
        // increasing order is increasing A index, so a strict < keeps the lowest chunk on ties
        const int npts = nch * kChunk;
        const int jbase = (chunk0 + k * C::kTileChunks) * kChunk;
        for (int e = tid; e < npts; e += kSymThreads) {
            const int j = jbase + e;
            if (j < p.nb) {
                unsigned m = cbuf[e];
                unsigned wbest = 0;
#pragma unroll
                for (int ws = 1; ws < kSymWarps * S; ++ws) {
                    const unsigned v = cbuf[ws * C::kTilePoints + e];
                    if (v < m) { m = v; wbest = (unsigned)ws; }
                }
                const u64 key = ((u64)m << 32) | (u64)(colchunk_base + wbest);
                if (p.qblocks == 1) keys_col[j] = key;
                else atomicMin(&keys_col[j], key);
                if (m < 0x7f800000u) cmax = max(cmax, m);
            }
        }
        // cbuf (k & 1) is rewritten in tile k+2, after the __syncthreads of tile k+1 which every thread reaches
        // only after finishing this fold
    }

    if (CULL && p.cull_stats && lane == 0) {                  // (warp, chunk) pairs evaluated / offered: the culling rate
        atomicAdd(p.cull_stats, (unsigned long long)evaluated);
        atomicAdd(p.cull_stats + 1, (unsigned long long)max(nchunks, 0));
    }
    if (p.col_bound) {                                       // one atomic per warp: bound for the fixed-point energy scatter
        cmax = __reduce_max_sync(0xffffffffu, cmax);
        if (lane == 0 && cmax) atomicMax(p.col_bound, cmax);
    }

    u64* __restrict__ keys_row = p.keys_a + (int64_t)b * p.na;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = qbase + warp * (32 * R) + (r / RS) * (32 * RS) + lane * RS + (r % RS);
        if (i < p.na) {
            const u64 key = ((u64)__float_as_uint(best[r]) << 32) | (u64)bch[r];
            if (p.splits == 1) keys_row[i] = key;
            else atomicMin(&keys_row[i], key);
        }
    }
}

// ----------------------------------------------------------------------------- culled search, warps decoupled
// The CULL instantiation above keeps the brute-force structure: a barrier per tile and a CTA-wide fold of the 8 warps'
// column minima.  Under culling that structure is the bottleneck: every warp skips DIFFERENT chunks, the barrier makes a
// tile cost the MAXIMUM of the 8 warps' surviving chunks, and measured time was 0.59 of the brute force at 0.35 of the
// blocks evaluated.  Here the warps of a CTA only share the TMA ring:
//   * a warp merges the column minima of a chunk it evaluated straight into the global keys -- one predicated 64-bit
//     atomicMin per lane (lane = target), and only when its value is <= the chunk's column bound (the final minimum of
//     every column of the chunk is <= that bound, so nothing larger can be a final minimum); skipped chunks merge nothing;
//   * no per-tile barrier: a warp that finished a tile bumps a per-stage counter, the LAST of the 8 re-arms the stage and
//     issues the next TMA into it, so the warps drift apart by up to kCullStages - 1 tiles and the per-tile maxima
//     average out.
// Same keys as the brute force, bit for bit (tests/test_cull_gpu.py).
//
// TIES = true also leaves a per-point TIE WORD (p.tie_a / p.tie_b, 0xffffffff on entry): the smallest distance, as bits, at
// which two DIFFERENT chunks were seen to reach the same value.  A search over a permuted copy of the clouds needs it: a
// key names the first chunk of the SEARCH order that reaches the minimum, while the caller's semantics is the lowest
// index of the CALLER's order, so a point whose minimum is reached in two chunks (tie word == final distance) must be
// resolved exactly by the consumer (energy.cu).  Detection is exact: a row folds every chunk into a chunk-local minimum
// (same min3 count as the running one) and compares it with the running minimum at the chunk's end; partial results of
// different work items meet through atomicMin, whose returned old value shows a tie -- of two minimum-attaining chunks,
// the one that merges second sees the first one's value.  A skipped chunk cannot hold a minimum (the skip test is strict).
constexpr int kCullStages = 6;
constexpr int kCullTileChunks = 16;
constexpr int kCullTileBytes = kCullTileChunks * kChunk * 12;
constexpr int kCullStageBytes = kCullTileBytes + kCullTileChunks * kBoxFloats * 4;

template <int NT, bool TIES>
__global__ void __launch_bounds__(NT, 512 / NT) chamfer_sym_cull_kernel(const SymParams p) {
    constexpr int kWarps = NT / 32;
    constexpr int R = 8;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[kCullStages];
    __shared__ unsigned done_cnt[kCullStages];

    int item = blockIdx.x;
    const int qb = item % p.qblocks;
    item /= p.qblocks;
    const int split = item % p.splits;
    const int b = item / p.splits;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int qbase = qb * (R * NT);
    const float* __restrict__ q = p.a + (int64_t)b * p.na * 3;

    const int chunks_total = p.nb_pad / kChunk;
    const int cps = (chunks_total + p.splits - 1) / p.splits;
    const int chunk0 = split * cps;
    const int nchunks = min(cps, chunks_total - chunk0);
    const int ntiles = (nchunks + kCullTileChunks - 1) / kCullTileChunks;
    const float* __restrict__ tp = p.b_packed + (int64_t)b * p.nb_pad * 3 + (int64_t)chunk0 * kChunk * 3;
    const float* __restrict__ bp = p.colbox + ((int64_t)b * chunks_total + chunk0) * kBoxFloats;
    u64* __restrict__ keys_col = p.keys_b + (int64_t)b * p.nb;
    const u64 colchunk = (u64)(qbase / 256 + warp);              // this warp's 256-row chunk: the column keys' low word

    auto issue = [&](int k) {
        const int st = k % kCullStages;
        const int nch = min(kCullTileChunks, nchunks - k * kCullTileChunks);
        const uint32_t bytes = (uint32_t)nch * kChunk * 12, box_bytes = (uint32_t)nch * kBoxFloats * 4;
        mbar_expect_tx(&full_bar[st], bytes + box_bytes);
        tma_bulk_g2s(smem_raw + st * kCullStageBytes, tp + (int64_t)k * kCullTileChunks * kChunk * 3, bytes, &full_bar[st]);
        tma_bulk_g2s(smem_raw + st * kCullStageBytes + kCullTileBytes, bp + (int64_t)k * kCullTileChunks * kBoxFloats, box_bytes,
                     &full_bar[st]);
    };
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kCullStages; ++s) { mbar_init(&full_bar[s], 1); done_cnt[s] = 0u; }
        mbar_fence_init();
        for (int k = 0; k < min(kCullStages, ntiles); ++k) issue(k);
    }

    u64 QX[R], QY[R], QZ[R];
    float best[R], prev[R];                                    // TIES: prev is the chunk-local minimum
    unsigned bch[R];
    unsigned tied = 0u;                                        // TIES: bit r = row r's running minimum is reached in two chunks
    float rlx = INFINITY, rly = INFINITY, rlz = INFINITY, rhx = -INFINITY, rhy = -INFINITY, rhz = -INFINITY;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = qbase + warp * (32 * R) + lane * R + r;
        float x = INFINITY, y = INFINITY, z = INFINITY;          // out-of-range rows never win a column
        if (i < p.na) {
            x = q[3 * i]; y = q[3 * i + 1]; z = q[3 * i + 2];
            rlx = fminf(rlx, x); rly = fminf(rly, y); rlz = fminf(rlz, z);
            rhx = fmaxf(rhx, x); rhy = fmaxf(rhy, y); rhz = fmaxf(rhz, z);
        }
        QX[r] = pack2(x, x); QY[r] = pack2(y, y); QZ[r] = pack2(z, z);
        best[r] = INFINITY; prev[r] = INFINITY; bch[r] = 0u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        rlx = fminf(rlx, __shfl_xor_sync(0xffffffffu, rlx, o)); rly = fminf(rly, __shfl_xor_sync(0xffffffffu, rly, o));
        rlz = fminf(rlz, __shfl_xor_sync(0xffffffffu, rlz, o)); rhx = fmaxf(rhx, __shfl_xor_sync(0xffffffffu, rhx, o));
        rhy = fmaxf(rhy, __shfl_xor_sync(0xffffffffu, rhy, o)); rhz = fmaxf(rhz, __shfl_xor_sync(0xffffffffu, rhz, o));
    }
    float rbound = INFINITY;
    {
        const int rc = qbase / (32 * R) + warp;
        if (rc * (32 * R) < p.na) rbound = __ldg(p.rowbound + (int64_t)b * p.row_chunks + rc);
    }
    unsigned evaluated = 0u, cmax = 0u;
    __syncthreads();                                         // barrier initialisation visible to every waiter

    for (int k = 0; k < ntiles; ++k) {
        const int st = k % kCullStages;
        mbar_wait(&full_bar[st], (uint32_t)((k / kCullStages) & 1));
        const int nch = min(kCullTileChunks, nchunks - k * kCullTileChunks);
        const float4* __restrict__ tile = reinterpret_cast<const float4*>(smem_raw + st * kCullStageBytes);
        const float* __restrict__ sbox = reinterpret_cast<const float*>(smem_raw + st * kCullStageBytes + kCullTileBytes);
        for (int c = 0; c < nch; ++c) {
            const float4 b0 = *reinterpret_cast<const float4*>(sbox + c * kBoxFloats);
            const float4 b1 = *reinterpret_cast<const float4*>(sbox + c * kBoxFloats + 4);
            // b0 = (lo.x, lo.y, lo.z, hi.x), b1 = (hi.y, hi.z, column bound, -)
            const float gx = fmaxf(0.f, fmaxf(__fsub_rn(rlx, b0.w), __fsub_rn(b0.x, rhx)));
            const float gy = fmaxf(0.f, fmaxf(__fsub_rn(rly, b1.x), __fsub_rn(b0.y, rhy)));
            const float gz = fmaxf(0.f, fmaxf(__fsub_rn(rlz, b1.y), __fsub_rn(b0.z, rhz)));
            const float lb = __fmaf_rn(gz, gz, __fmaf_rn(gy, gy, __fmul_rn(gx, gx)));
            if (lb > rbound && lb > b1.z) continue;            // warp-uniform: no minimum and no tie of either side in here
            ++evaluated;
            const float4* __restrict__ cg = tile + c * (kChunk / 4 * 3);
            unsigned mine = 0x7f800000u;                       // the warp's minimum for target (this lane) of the chunk
            if (TIES) {
#pragma unroll
                for (int r = 0; r < R; ++r) prev[r] = INFINITY;
            }
#pragma unroll
            for (int g = 0; g < kChunk / 4; ++g) {
                const float4 X = cg[3 * g], Y = cg[3 * g + 1], Z = cg[3 * g + 2];
                const u64 X01 = pack2(X.x, X.y), X23 = pack2(X.z, X.w);
                const u64 Y01 = pack2(Y.x, Y.y), Y23 = pack2(Y.z, Y.w);
                const u64 Z01 = pack2(Z.x, Z.y), Z23 = pack2(Z.z, Z.w);
                float c0, c1, c2, c3;
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    float a0, a1, a2, a3;
                    unpack2(sqdist_pair(QX[r], QY[r], QZ[r], X01, Y01, Z01), a0, a1);
                    unpack2(sqdist_pair(QX[r], QY[r], QZ[r], X23, Y23, Z23), a2, a3);
                    float& acc = TIES ? prev[r] : best[r];
                    acc = min3(acc, a0, a1);
                    acc = min3(acc, a2, a3);
                    if (r == 0) { c0 = a0; c1 = a1; c2 = a2; c3 = a3; }
                    else { c0 = fminf(c0, a0); c1 = fminf(c1, a1); c2 = fminf(c2, a2); c3 = fminf(c3, a3); }
                }
                const unsigned m0 = __reduce_min_sync(0xffffffffu, __float_as_uint(c0));
                const unsigned m1 = __reduce_min_sync(0xffffffffu, __float_as_uint(c1));
                const unsigned m2 = __reduce_min_sync(0xffffffffu, __float_as_uint(c2));
                const unsigned m3 = __reduce_min_sync(0xffffffffu, __float_as_uint(c3));
                if ((lane >> 2) == g) mine = (lane & 2) ? ((lane & 1) ? m3 : m2) : ((lane & 1) ? m1 : m0);
            }
            const unsigned gid = (unsigned)(chunk0 + k * kCullTileChunks + c);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (TIES) {
                    if (prev[r] < best[r]) { best[r] = prev[r]; bch[r] = gid; tied &= ~(1u << r); }
                    else if (prev[r] == best[r]) tied |= 1u << r;
                } else {
                    if (best[r] < prev[r]) bch[r] = gid;
                    prev[r] = best[r];
                }
            }
            const int j = (int)gid * kChunk + lane;
            if (j < p.nb && mine <= __float_as_uint(b1.z)) {   // <=: a tie with the bound can still be the final minimum
                const u64 old = atomicMin(&keys_col[j], ((u64)mine << 32) | colchunk);
                if (TIES && (unsigned)(old >> 32) == mine) atomicMin(p.tie_b + (int64_t)b * p.nb + j, mine);   // another row chunk
                if (mine < 0x7f800000u) cmax = max(cmax, mine);
            }
        }
        // this warp is done with the stage; the last of the 8 warps re-arms it and requests the tile that reuses it
        __syncwarp();
        if (lane == 0) {
            __threadfence_block();
            if (atomicAdd(&done_cnt[st], 1u) == (unsigned)(kWarps - 1)) {
                done_cnt[st] = 0u;
                __threadfence_block();
                if (k + kCullStages < ntiles) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    issue(k + kCullStages);
                }
            }
        }
    }

    if (p.cull_stats && lane == 0) {
        atomicAdd(p.cull_stats, (unsigned long long)evaluated);
        atomicAdd(p.cull_stats + 1, (unsigned long long)max(nchunks, 0));
    }
    if (p.col_bound) {
        cmax = __reduce_max_sync(0xffffffffu, cmax);
        if (lane == 0 && cmax) atomicMax(p.col_bound, cmax);
    }
    u64* __restrict__ keys_row = p.keys_a + (int64_t)b * p.na;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = qbase + warp * (32 * R) + lane * R + r;
        if (i < p.na) {
            const unsigned d = __float_as_uint(best[r]);
            const u64 key = ((u64)d << 32) | (u64)bch[r];
            unsigned tie = ((tied >> r) & 1u) ? d : 0xffffffffu;
            if (p.splits == 1) {
                keys_row[i] = key;
            } else {
                const u64 old = atomicMin(&keys_row[i], key);
                if (TIES && (unsigned)(old >> 32) == d) tie = d;     // the other split's chunks are different chunks
            }
            if (TIES && tie != 0xffffffffu) atomicMin(p.tie_a + (int64_t)b * p.na + i, tie);
        }
    }
}

// (Measured and rejected in round 2: a persistent one-wave schedule that gives each of 2 x 148 CTAs an equal contiguous
// share of the (row block, chunk) units -- 3.98 ms instead of 3.69 ms at 64 frames, 0.520 instead of 0.499 ms at 8: with
// equal static shares the slowest CTA sets the time, while one CTA per item lets the hardware scheduler absorb the
// SM-to-SM variance.  profiles/r02_scaling.md.)
// Number of target splits per (frame, query block).  CTAs map 1:1 to work items and two are resident per SM, so
// the grid runs in waves of 2*148 CTAs: pick the split count whose item total wastes the least of its last wave
// (strong scaling leaves few frames per GPU, where a bad count costs 15-25 % of the kernel), preferring fewer,
// larger items on ties, and keeping at least one full tile (512 targets) per item.
static int sym_choose_splits(int64_t B, int qblocks, int chunks_total, int tile_chunks) {
    const int64_t slots = 2 * 148;
    const int64_t base = std::max<int64_t>(1, B * qblocks);
    // normally at least one full tile (512 targets) per item; when even that leaves SMs idle go down to 128 targets
    int max_s = std::max(1, chunks_total / std::max(tile_chunks, 16));
    if (base * max_s < slots) max_s = std::max(max_s, chunks_total / 4);
    if (base >= 8 * slots) return 1;                        // plenty of items already: tail < 1/8 wave
    int best_s = 1;
    double best_eff = -1.0;
    for (int sp = 1; sp <= max_s; ++sp) {
        const int64_t items = base * sp;
        const int64_t waves = ceil_div(items, slots);
        double eff = (double)items / (double)(waves * slots);
        if (waves >= 8) eff = std::max(eff, 0.97);         // many waves: the tail no longer matters
        // each item pays a fixed prologue/epilogue (~2 % of a 1024-target item): charge it
        const double per_item_targets = (double)chunks_total * kChunk / sp;
        eff *= per_item_targets / (per_item_targets + 24.0);
        if (eff > best_eff + 1e-9) { best_eff = eff; best_s = sp; }
    }
    return best_s;
}

template <int R, int S, bool CULL, bool SKIN = false>
static int launch_sym_rs(SymParams& p, cudaStream_t stream) {
    using C = SymCfg<R, S>;
    p.qblocks = (int)ceil_div(p.na, R * kSymThreads);
    p.splits = sym_choose_splits(p.B, p.qblocks, p.nb_pad / kChunk, C::kTileChunks);
    if (p.variant >= 16) p.splits = std::max(1, std::min(p.variant / 16, p.nb_pad / kChunk));   // tuning override
    p.col_chunk_pts = C::kColChunkPts;
    const int64_t items = (int64_t)p.B * p.qblocks * p.splits;
    if (items <= 0) return kOk;
    if (items > 0x7fffffff) return kErrUnsupported;
    // merge keys start at +max wherever partial results meet through atomicMin; one memset when the two arrays are
    // neighbours in the workspace (they are in every pipeline of capi.cu)
    const bool need_a = p.splits > 1 && !p.keys_preset, need_b = p.qblocks > 1 && !p.keys_preset;
    const size_t bytes_a = sizeof(u64) * (size_t)p.B * p.na, bytes_b = sizeof(u64) * (size_t)p.B * p.nb;
    const char* a0 = reinterpret_cast<const char*>(p.keys_a);
    const char* b0 = reinterpret_cast<const char*>(p.keys_b);
    // (one memset may only span the gap between the two arrays when both live in ONE allocation of ours -- the fused
    // pipelines of capi.cu say so with keys_one_allocation; caller-owned arrays may have a stranger's tensor in between)
    if (p.keys_one_allocation && need_a && need_b && b0 >= a0 + bytes_a && (size_t)(b0 - a0) <= bytes_a + 4096) {
        if (cudaMemsetAsync(p.keys_a, 0xff, (size_t)(b0 - a0) + bytes_b, stream) != cudaSuccess) return kErrLaunch;
    } else {
        if (need_a && cudaMemsetAsync(p.keys_a, 0xff, bytes_a, stream) != cudaSuccess) return kErrLaunch;
        if (need_b && cudaMemsetAsync(p.keys_b, 0xff, bytes_b, stream) != cudaSuccess) return kErrLaunch;
    }
    // opt in to > 48 KB dynamic shared memory once per device (not a stream operation; safe under graph capture)
    static bool attr_done[64] = {};
    int devid = 0;
    cudaGetDevice(&devid);
    if (devid < 0 || devid >= 64 || !attr_done[devid]) {
        if (cudaFuncSetAttribute(chamfer_sym_kernel<R, S, CULL, SKIN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(C::kSmem + kSymStages * C::kTileChunks * kBoxFloats * 4)) != cudaSuccess)
            return kErrLaunch;
        if (devid >= 0 && devid < 64) attr_done[devid] = true;
    }
    const size_t smem = C::kSmem + (CULL ? (size_t)kSymStages * C::kTileChunks * kBoxFloats * 4 : 0);
    chamfer_sym_kernel<R, S, CULL, SKIN><<<(unsigned)items, kSymThreads, smem, stream>>>(p);
    REART_CHECK_LAUNCH();
    return kOk;
}

static int launch_sym_cull(SymParams& p, cudaStream_t stream) {
    using C = SymCfg<8, 1>;
    const int nt = (p.variant == 2) ? 256 : 128;               // 4 warps per CTA, 4 CTAs per SM: less idle time at the end of an item
    p.qblocks = (int)ceil_div(p.na, 8 * nt);
    {
        // item durations vary with what survives the culling, so wave arithmetic is moot: aim at ~8 items per CTA slot for
        // the hardware scheduler to balance, but keep >= 2 tiles per item (prologue amortised, room for the warps to drift)
        const int64_t slots = (int64_t)(512 / nt) * 148, base = std::max<int64_t>(1, (int64_t)p.B * p.qblocks);
        const int chunks_total = p.nb_pad / kChunk;
        const int64_t want = ceil_div(8 * slots, base), cap = std::max(1, chunks_total / (2 * kCullTileChunks));
        p.splits = (int)std::max<int64_t>(1, std::min(want, cap));
    }
    p.col_chunk_pts = C::kColChunkPts;
    const int64_t items = (int64_t)p.B * p.qblocks * p.splits;
    if (items <= 0) return kOk;
    if (items > 0x7fffffff) return kErrUnsupported;
    if (p.tie_a && cudaMemsetAsync(p.tie_a, 0xff, sizeof(unsigned) * (size_t)p.B * (p.na + p.nb), stream) != cudaSuccess)
        return kErrLaunch;                                     // [tie_a | tie_b] are one array
    if (!p.keys_preset) {
        // every column key is merged by atomicMin here (no CTA-level fold), row keys when the targets are split
        const size_t bytes_a = sizeof(u64) * (size_t)p.B * p.na, bytes_b = sizeof(u64) * (size_t)p.B * p.nb;
        const char* a0 = reinterpret_cast<const char*>(p.keys_a);
        const char* b0 = reinterpret_cast<const char*>(p.keys_b);
        if (p.keys_one_allocation && p.splits > 1 && b0 >= a0 + bytes_a && (size_t)(b0 - a0) <= bytes_a + 4096) {
            if (cudaMemsetAsync(p.keys_a, 0xff, (size_t)(b0 - a0) + bytes_b, stream) != cudaSuccess) return kErrLaunch;
        } else {
            if (p.splits > 1 && cudaMemsetAsync(p.keys_a, 0xff, bytes_a, stream) != cudaSuccess) return kErrLaunch;
            if (cudaMemsetAsync(p.keys_b, 0xff, bytes_b, stream) != cudaSuccess) return kErrLaunch;
        }
    }
    const size_t smem = (size_t)kCullStages * kCullStageBytes;
    if (p.tie_a) {
        if (nt == 256) chamfer_sym_cull_kernel<256, true><<<(unsigned)items, 256, smem, stream>>>(p);
        else chamfer_sym_cull_kernel<128, true><<<(unsigned)items, 128, smem, stream>>>(p);
    } else {
        if (nt == 256) chamfer_sym_cull_kernel<256, false><<<(unsigned)items, 256, smem, stream>>>(p);
        else chamfer_sym_cull_kernel<128, false><<<(unsigned)items, 128, smem, stream>>>(p);
    }
    REART_CHECK_LAUNCH();
    return kOk;
}

int launch_chamfer_sym(SymParams& p, cudaStream_t stream) {
    // Measured on B200 (profiles/r01_sym_variants.log, T=64 x 16k): S=1 3.70 ms, S=2 3.87, S=4 4.17, S=8 4.45 --
    // one REDUX per target (S=1, 256-point column chunks) is the fastest search even after paying for the wider
    // index recovery (which the x-sorted packed copy makes cheap, skin.cu / energy.cu).
    if (p.sk_cano) {                                           // fused producer (one-hot weights in compact form)
        if (p.cull || !p.sk_hot || !p.sk_R || !p.sk_tr || !p.sk_out || !p.sk_sorted || !p.sk_perm || !p.sk_xq ||
            p.sk_P <= 0 || p.sk_P > 32 || p.sk_npad % 256 != 0 || p.sk_npad < p.na)
            return kErrInvalidArg;
        return launch_sym_rs<8, 1, false, true>(p, stream);
    }
    if (p.cull) {
        if (!p.colbox || !p.rowbound || (p.tie_a && p.tie_b != p.tie_a + (int64_t)p.B * p.na)) return kErrInvalidArg;
        p.row_chunks = (int)ceil_div(p.na, 256);
        if (p.variant == 1) return launch_sym_rs<8, 1, true>(p, stream);      // the barrier-per-tile culled kernel (comparison)
        return launch_sym_cull(p, stream);
    }
    switch (p.variant % 16) {
        case 2: return launch_sym_rs<8, 2, false>(p, stream);
        case 4: return launch_sym_rs<8, 4, false>(p, stream);
        case 8: return launch_sym_rs<8, 8, false>(p, stream);
        default: return launch_sym_rs<8, 1, false>(p, stream);
    }
}

}  // namespace reart
