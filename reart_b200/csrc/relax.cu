// relax.cu -- the FRAME-INDEPENDENT part of one relaxation iteration (run_robot.py:154-221, --model=base), fused into
// one "head" and one "tail" kernel.  Under frame sharding everything else in a step shrinks with the number of GPUs;
// this part does not, so it bounds strong scaling (VERDICT r01: ~12 launches, 0.09 ms of a 0.69 ms step at 8 GPUs).
//
//   head  = seg MLP forward (networks/blocks.py:99-118 as built at networks/model.py:19,42-43)
//           + straight-through gumbel-softmax weights from torch-drawn Exponential(1) noise (networks/model.py:44)
//           + 6D -> R for every (frame, part) (networks/model.py:60, screw_se3/geo_utils.py:632-651);
//   tail  = gumbel backward + seg MLP backward (per-chunk partials, summed in a FIXED order by the last block)
//           + 6D backward + [the one-shot all-reduce of allreduce.cu, inline, when frames are sharded]
//           + Adam (torch.optim.Adam semantics, run_robot.py:146-150,219-221) on all five parameter tensors.
// No float atomics anywhere: every sum has a fixed association, so a step is bit-reproducible.
#include "common.cuh"
#include "kernels.h"
#include "se3_device.cuh"
#include "tail_device.cuh"
#include <algorithm>
#include <cmath>

namespace reart {

// ============================================================================================ head
constexpr int kHeadThreads = 256;                            // kMlpLanes = 8 lanes per point -> 32 points per block

template <int PMAX>
__global__ void __launch_bounds__(kHeadThreads) relax_head_kernel(const float* __restrict__ x,
                                                                  const float* __restrict__ w0,
                                                                  const float* __restrict__ b0,
                                                                  const float* __restrict__ w2,
                                                                  const float* __restrict__ expo,
                                                                  const int64_t* __restrict__ noise_index,
                                                                  const float* __restrict__ tau_ptr,
                                                                  const float* __restrict__ d6, int N, int H, int P,
                                                                  int TP, int point_blocks, float* __restrict__ logits,
                                                                  float* __restrict__ W, float* __restrict__ ysoft,
                                                                  float* __restrict__ R, float* __restrict__ hot_out) {
    if ((int)blockIdx.x >= point_blocks) {                    // trailing blocks: 6D -> R, one thread per (frame, part)
        const int i = ((int)blockIdx.x - point_blocks) * kHeadThreads + threadIdx.x;
        if (i < TP) {
            float in[6], out[9];
#pragma unroll
            for (int k = 0; k < 6; ++k) in[k] = d6[(int64_t)i * 6 + k];
            rot6d_eval<float>(in, out);
#pragma unroll
            for (int k = 0; k < 9; ++k) R[(int64_t)i * 9 + k] = out[k];
        }
        return;
    }
    extern __shared__ __align__(16) float sm[];
    float* s0 = sm;                       // [H][4]: w0 row + bias
    float* s2 = sm + H * 4;               // [H][PMAX + 4]: W2 transposed, zero padded
    segmlp_stage<PMAX>(w0, b0, w2, H, P, s0, s2);
    __syncthreads();
    // seg MLP: kMlpLanes lanes per point (the function segmlp_fwd_kernel uses, so both paths give the same logits)
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = gid / kMlpLanes, part = gid % kMlpLanes;
    const bool real = n < N;
    float px = 0.f, py = 0.f, pz = 0.f;
    if (real) { px = x[3 * n]; py = x[3 * n + 1]; pz = x[3 * n + 2]; }
    float acc[PMAX];
    segmlp_point<PMAX>(s0, s2, H, part, px, py, pz, acc);
    // straight-through gumbel softmax.  The transcendental work is SPLIT over the point's lanes (lane l evaluates the
    // parts p = l, l + kMlpLanes, ...), the values are gathered back with shuffles and then summed / compared in part
    // order by every lane -- the arithmetic and its order are those of gumbel_st_kernel, so W and ysoft agree bit for bit.
    const float inv_tau = 1.0f / *tau_ptr;
    // noise row of this point: its own, or (point order changed by the caller, e.g. the engine's k-d order) the row the
    // point had in the order the noise was drawn for -- the optimisation then takes the same random decisions
    const int64_t nrow = real ? (noise_index ? noise_index[n] : (int64_t)n) : 0;
    constexpr int kOwn = (PMAX + kMlpLanes - 1) / kMlpLanes;
    float zown[kOwn];
    float mx = -INFINITY;
#pragma unroll
    for (int q = 0; q < kOwn; ++q) {
        const int p = part + q * kMlpLanes;
        zown[q] = -INFINITY;
        if (real && p < P) {
            float a = 0.f;
#pragma unroll
            for (int pp = 0; pp < PMAX; ++pp) if (pp == p) a = acc[pp];           // register select (no dynamic indexing)
            zown[q] = (a - logf(expo[nrow * P + p])) * inv_tau;
            mx = fmaxf(mx, zown[q]);
        }
    }
#pragma unroll
    for (int o = 1; o < kMlpLanes; o <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
#pragma unroll
    for (int q = 0; q < kOwn; ++q) zown[q] = expf(zown[q] - mx);                   // -inf slots -> 0, never read
    const int lane0 = (threadIdx.x & 31) & ~(kMlpLanes - 1);                      // first lane of this point's group
    float z[PMAX];
    float sum = 0.f;
#pragma unroll
    for (int p = 0; p < PMAX; ++p) {
        const float v = __shfl_sync(0xffffffffu, zown[p / kMlpLanes], lane0 + (p % kMlpLanes));
        z[p] = v;
        if (p < P) sum += v;
    }
    int hot = 0;
    float best = -1.f;
#pragma unroll
    for (int p = 0; p < PMAX; ++p)
        if (p < P) { z[p] = z[p] / sum; if (z[p] > best) { best = z[p]; hot = p; } }
    if (!real) return;
#pragma unroll
    for (int p = 0; p < PMAX; ++p) {
        if (p < P && (p % kMlpLanes) == part) {
            const float y = z[p];
            if (logits) logits[(int64_t)n * P + p] = acc[p];
            ysoft[(int64_t)n * P + p] = y;
            const float wv = ((p == hot ? 1.0f : 0.0f) - y) + y;
            W[(int64_t)n * P + p] = wv;
            // the row's ONE non-zero in compact form for the fused producer of the search (every other entry is (0 - y) + y = 0)
            if (hot_out && p == hot) reinterpret_cast<int2*>(hot_out)[n] = make_int2(hot, __float_as_int(wv));
        }
    }
}

int launch_relax_head(const float* cano, const float* w0, const float* b0, const float* w2, const float* expo,
                      const int64_t* noise_index, const float* tau, const float* d6, int64_t N, int64_t H, int64_t P, int64_t T, float* logits,
                      float* W, float* ysoft, float* R, float* hot, cudaStream_t stream) {
    if (N <= 0 && T <= 0) return kOk;
    if (H <= 0 || H > 1024 || P <= 0 || P > 32) return kErrUnsupported;
    const int point_blocks = (int)ceil_div(kMlpLanes * N, kHeadThreads);
    const int pose_blocks = (int)ceil_div(T * P, kHeadThreads);
#define REART_HEAD(PM)                                                                                               \
    do {                                                                                                             \
        const size_t smem = (size_t)H * (4 + PM + 4) * sizeof(float);                                                \
        if (smem > 48 * 1024) return kErrUnsupported;                                                                \
        relax_head_kernel<PM><<<(unsigned)(point_blocks + pose_blocks), kHeadThreads, smem, stream>>>(               \
            cano, w0, b0, w2, expo, noise_index, tau, d6, (int)N, (int)H, (int)P, (int)(T * P), point_blocks, logits, W, ysoft, R, hot); \
    } while (0)
    if (P <= 8) REART_HEAD(8);
    else if (P <= 16) REART_HEAD(16);
    else REART_HEAD(32);
#undef REART_HEAD
    REART_CHECK_LAUNCH();
    return kOk;
}

// ============================================================================================ tail
constexpr int kTailPoints = 128;                             // points per block (seg-MLP backward chunk)
constexpr int kTailGroup = 8;                                // chunks per first-level reduction group

// grid = point_blocks (128 points each) + pose_blocks; threads = 4 * Hpad  (Hpad = H rounded up to 32, <= 256)
template <int PMAX>
__global__ void __launch_bounds__(1024) relax_tail_kernel(const RelaxTail a, int point_blocks, int Hpad) {
    extern __shared__ __align__(16) float sm[];
    __shared__ bool last_pts, last_grp;
    __shared__ int s_ok;
    const int tid = threadIdx.x;
    const int H = a.H, P = a.P;
    const int nseg = 4 * H + P * H;
    const float step = *a.step + 1.0f;                        // 1-based index of this optimisation step

    if ((int)blockIdx.x >= point_blocks) {
        // ------------------------------------------------ pose side: 6D backward + Adam on proposal_6d / proposal_t
        if (a.phase != 1) {
            const int i = ((int)blockIdx.x - point_blocks) * blockDim.x + tid;
            if (i < a.T * P) {
                const AdamCoef c = adam_coef(a.lr_pose, a.beta1, a.beta2, a.eps, a.wd, step);
                Dual<6> in[6], out[9];
#pragma unroll
                for (int k = 0; k < 6; ++k) in[k] = Dual<6>::var(a.d6[(int64_t)i * 6 + k], k);
                rot6d_eval<Dual<6>>(in, out);
                float g[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int o = 0; o < 9; ++o) {
                    const float go = a.gR[(int64_t)i * 9 + o];
#pragma unroll
                    for (int k = 0; k < 6; ++k) g[k] += go * out[o].d[k];
                }
#pragma unroll
                for (int k = 0; k < 6; ++k) adam_update(a.d6 + (int64_t)i * 6 + k, a.m_d6 + (int64_t)i * 6 + k, a.v_d6 + (int64_t)i * 6 + k, g[k], c);
#pragma unroll
                for (int k = 0; k < 3; ++k) adam_update(a.tr + (int64_t)i * 3 + k, a.m_tr + (int64_t)i * 3 + k, a.v_tr + (int64_t)i * 3 + k, a.gtr[(int64_t)i * 3 + k], c);
            }
        }
    } else if (a.phase != 2) {
        // ------------------------------------------------ point side: gumbel backward + seg MLP backward of one chunk
        float* sx = sm;                                       // [kTailPoints][4]
        float* sg = sx + kTailPoints * 4;                     // [kTailPoints][PMAX]  d loss / d logits
        float* sred = sg + kTailPoints * PMAX;                // [3][Hpad][4 + PMAX]
        const int n0 = blockIdx.x * kTailPoints;
        const int cnt = min(kTailPoints, a.N - n0);
        const float inv_tau = 1.0f / *a.tau;
        for (int e = tid; e < kTailPoints; e += blockDim.x) {
            const bool ok = e < cnt;
            sx[4 * e] = ok ? a.cano[3 * (n0 + e)] : 0.f; sx[4 * e + 1] = ok ? a.cano[3 * (n0 + e) + 1] : 0.f;
            sx[4 * e + 2] = ok ? a.cano[3 * (n0 + e) + 2] : 0.f; sx[4 * e + 3] = 0.f;
            // dL/dlogits = y * (g - sum_p g_p y_p) / tau   (straight-through: the hard part has no gradient)
            float dot = 0.f;
            if (ok) {
#pragma unroll
                for (int p = 0; p < PMAX; ++p)
                    if (p < P) dot += a.gW[(int64_t)(n0 + e) * P + p] * a.ysoft[(int64_t)(n0 + e) * P + p];
            }
#pragma unroll
            for (int p = 0; p < PMAX; ++p) {
                float v = 0.f;
                if (ok && p < P) {
                    const float y = a.ysoft[(int64_t)(n0 + e) * P + p];
                    v = y * (a.gW[(int64_t)(n0 + e) * P + p] - dot) * inv_tau;
                }
                sg[e * PMAX + p] = v;
            }
        }
        __syncthreads();
        // thread = (hidden unit k, point quarter q): sums over its 32 points stay in registers
        const int k = tid % Hpad, q = tid / Hpad;
        const bool unit = k < H;
        float wx = 0.f, wy = 0.f, wz = 0.f, bb = 0.f;
        float w2k[PMAX], a2[PMAX];
#pragma unroll
        for (int p = 0; p < PMAX; ++p) { w2k[p] = 0.f; a2[p] = 0.f; }
        if (unit) {
            wx = a.w0[3 * k]; wy = a.w0[3 * k + 1]; wz = a.w0[3 * k + 2]; bb = a.b0[k];
#pragma unroll
            for (int p = 0; p < PMAX; ++p) if (p < P) w2k[p] = a.w2[p * H + k];
        }
        float ax = 0.f, ay = 0.f, az = 0.f, ab = 0.f;
        if (unit) {
            const int i0 = q * (kTailPoints / 4);
            for (int ii = 0; ii < kTailPoints / 4; ++ii) {
                const int i = i0 + ii;
                const float4 pt = reinterpret_cast<const float4*>(sx)[i];
                const float pre = wx * pt.x + wy * pt.y + wz * pt.z + bb;
                const float h = fmaxf(pre, 0.f);
                const float4* g4 = reinterpret_cast<const float4*>(sg + i * PMAX);
                float gh = 0.f;
#pragma unroll
                for (int r = 0; r < PMAX / 4; ++r) {
                    const float4 g = g4[r];
                    a2[4 * r] += g.x * h; a2[4 * r + 1] += g.y * h; a2[4 * r + 2] += g.z * h; a2[4 * r + 3] += g.w * h;
                    gh += g.x * w2k[4 * r] + g.y * w2k[4 * r + 1] + g.z * w2k[4 * r + 2] + g.w * w2k[4 * r + 3];
                }
                if (pre > 0.f) { ax += gh * pt.x; ay += gh * pt.y; az += gh * pt.z; ab += gh; }
            }
        }
        if (unit && q > 0) {
            float* o = sred + ((q - 1) * Hpad + k) * (4 + PMAX);
            o[0] = ax; o[1] = ay; o[2] = az; o[3] = ab;
#pragma unroll
            for (int p = 0; p < PMAX; ++p) o[4 + p] = a2[p];
        }
        __syncthreads();
        if (unit && q == 0) {                                  // quarters added in order 0,1,2,3
#pragma unroll
            for (int qq = 0; qq < 3; ++qq) {
                const float* o = sred + (qq * Hpad + k) * (4 + PMAX);
                ax += o[0]; ay += o[1]; az += o[2]; ab += o[3];
#pragma unroll
                for (int p = 0; p < PMAX; ++p) a2[p] += o[4 + p];
            }
            float* out = a.partials + (int64_t)blockIdx.x * nseg;
            out[3 * k] = ax; out[3 * k + 1] = ay; out[3 * k + 2] = az;
            out[3 * H + k] = ab;
#pragma unroll
            for (int p = 0; p < PMAX; ++p)
                if (p < P) out[4 * H + p * H + k] = a2[p];
        }
        __syncthreads();
        // ---- two-level fixed-order reduction of the per-chunk partials (a single last block summing all of them is a
        // chain of ~80 dependent L2 round trips at 128 chunks: 40 us).  Level 1: the last of each group of kTailGroup
        // consecutive chunks adds the group's partials in chunk order; level 2: the last group adds the group sums in
        // group order.  Both orders are fixed, so the bucket is bit-reproducible.
        const int ngroups = (point_blocks + kTailGroup - 1) / kTailGroup;
        const int grp = (int)blockIdx.x / kTailGroup;
        const int g0 = grp * kTailGroup, gn = min(kTailGroup, point_blocks - g0);
        float* gpart = a.partials + (int64_t)point_blocks * nseg;             // [ngroups][nseg]
        if (tid == 0) {
            __threadfence();
            last_grp = atomicAdd(a.tickets + 2 + grp, 1u) == (unsigned)gn - 1u;
        }
        __syncthreads();
        last_pts = false;
        if (last_grp) {
            __threadfence();
            const float* part = a.partials + (int64_t)g0 * nseg;
            if ((nseg & 3) == 0) {                              // four outputs per thread and load: fewer dependent round trips
                const int n4 = nseg >> 2;
                for (int e = tid; e < n4; e += blockDim.x) {
                    float4 v[kTailGroup];
#pragma unroll
                    for (int c = 0; c < kTailGroup; ++c)
                        v[c] = c < gn ? __ldcg(reinterpret_cast<const float4*>(part + (int64_t)c * nseg) + e) : make_float4(0.f, 0.f, 0.f, 0.f);
                    float4 sacc = v[0];
#pragma unroll
                    for (int c = 1; c < kTailGroup; ++c) { sacc.x += v[c].x; sacc.y += v[c].y; sacc.z += v[c].z; sacc.w += v[c].w; }
                    reinterpret_cast<float4*>(gpart + (int64_t)grp * nseg)[e] = sacc;
                }
            } else {
                for (int e = tid; e < nseg; e += blockDim.x) {
                    float v[kTailGroup];
#pragma unroll
                    for (int c = 0; c < kTailGroup; ++c) v[c] = c < gn ? __ldcg(part + (int64_t)c * nseg + e) : 0.f;
                    float sacc = v[0];
#pragma unroll
                    for (int c = 1; c < kTailGroup; ++c) sacc += v[c];
                    gpart[(int64_t)grp * nseg + e] = sacc;
                }
            }
            __syncthreads();
            if (tid == 0) {
                __threadfence();
                last_pts = atomicAdd(a.tickets, 1u) == (unsigned)ngroups - 1u;
            }
            __syncthreads();
        }
        if (last_pts) {
            // ---- the last group to finish: group sums -> bucket in group order, then [all-reduce], then Adam
            __threadfence();
            if ((nseg & 3) == 0) {
                const int n4 = nseg >> 2;
                for (int e = tid; e < n4; e += blockDim.x) {
                    float4 sacc = make_float4(0.f, 0.f, 0.f, 0.f);
                    for (int c = 0; c < ngroups; c += 16) {      // 16 loads in flight, added in group order
                        float4 v[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            v[i] = c + i < ngroups ? __ldcg(reinterpret_cast<const float4*>(gpart + (int64_t)(c + i) * nseg) + e)
                                                   : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                        for (int i = 0; i < 16; ++i) { sacc.x += v[i].x; sacc.y += v[i].y; sacc.z += v[i].z; sacc.w += v[i].w; }
                    }
                    reinterpret_cast<float4*>(a.bucket)[e] = sacc;
                }
            } else {
                for (int e = tid; e < nseg; e += blockDim.x) {
                    float sacc = 0.f;
                    for (int c = 0; c < ngroups; c += 16) {
                        float v[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = c + i < ngroups ? __ldcg(gpart + (int64_t)(c + i) * nseg + e) : 0.f;
#pragma unroll
                        for (int i = 0; i < 16; ++i) sacc += v[i];
                    }
                    a.bucket[e] = sacc;
                }
            }
            if (tid == 0) a.bucket[nseg] = (float)*reinterpret_cast<const volatile double*>(a.loss_local);
            __syncthreads();
        }
    }
    if (a.phase == 1) {                                        // reduce only: the caller all-reduces the bucket (NCCL)
        if ((int)blockIdx.x < point_blocks && last_pts) {       // re-arm the point-side tickets for the next launch
            const int ngroups = (point_blocks + kTailGroup - 1) / kTailGroup;
            for (int e = tid; e < ngroups; e += blockDim.x) a.tickets[2 + e] = 0u;
            if (tid == 0) a.tickets[0] = 0u;
        }
        return;
    }
    const bool seg_owner = a.phase == 2 ? (blockIdx.x == 0) : ((int)blockIdx.x < point_blocks && last_pts);
    if (seg_owner) {
        if (a.phase == 0 && a.world > 1)
            cta_allreduce_oneshot(a.peer_base, a.rank, a.world, nseg + 1, a.n_pad, a.epoch, a.bucket, &s_ok);
        const AdamCoef c = adam_coef(a.lr_seg, a.beta1, a.beta2, a.eps, a.wd, step);
        for (int e = tid; e < nseg; e += blockDim.x) {
            float* prm = e < 3 * H ? a.w0 + e : (e < 4 * H ? a.b0 + (e - 3 * H) : a.w2 + (e - 4 * H));
            adam_update(prm, a.m_seg + e, a.v_seg + e, a.bucket[e], c);
        }
        if (tid == 0) *a.loss_out = a.bucket[nseg];
    }
    // ---- the very last block of the launch (all roles) advances the step counter and re-arms the tickets
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(a.tickets + 1, 1u) == gridDim.x - 1u) {
            *a.step = step;
            const int ngroups = (point_blocks + kTailGroup - 1) / kTailGroup;
            for (int e = 0; e < 2 + ngroups; ++e) a.tickets[e] = 0u;
        }
    }
}

int64_t relax_tail_workspace_floats(int64_t N, int64_t H, int64_t P) {
    const int64_t blocks = ceil_div(N > 0 ? N : 1, kTailPoints);
    return (blocks + ceil_div(blocks, kTailGroup)) * (4 * H + P * H);
}
int64_t relax_tail_ticket_words(int64_t N) {
    return 2 + ceil_div(ceil_div(N > 0 ? N : 1, kTailPoints), kTailGroup);
}

int launch_relax_tail(const RelaxTail& a, cudaStream_t stream) {
    if (a.N <= 0 || a.T <= 0) return kErrInvalidArg;
    if (a.H <= 0 || a.H > 256 || a.P <= 0 || a.P > 32) return kErrUnsupported;
    const int Hpad = (int)round_up(a.H, 32);
    const int threads = 4 * Hpad;
    const int point_blocks = (int)ceil_div(a.N, kTailPoints);
    const int pose_blocks = (int)ceil_div((int64_t)a.T * a.P, threads);
    if (a.world > 1 && a.phase == 0 && (a.world > threads || !a.peer_base || !a.epoch)) return kErrInvalidArg;
    // smem grows with H (through Hpad), so the >48 KB opt-in is made once per device for the instantiation's LARGEST
    // launch (Hpad = 256): a later call with a larger H than the first must not exceed what was opted in
#define REART_TAIL(PM)                                                                                                 \
    do {                                                                                                               \
        const size_t smem = ((size_t)kTailPoints * (4 + PM) + (size_t)3 * Hpad * (4 + PM)) * sizeof(float);           \
        const size_t smem_max = ((size_t)kTailPoints * (4 + PM) + (size_t)3 * 256 * (4 + PM)) * sizeof(float);        \
        static bool attr_done[64] = {};                                                                                \
        int devid = 0;                                                                                                 \
        cudaGetDevice(&devid);                                                                                         \
        if (smem > 48 * 1024 && (devid < 0 || devid >= 64 || !attr_done[devid])) {                                     \
            if (cudaFuncSetAttribute(relax_tail_kernel<PM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max) != cudaSuccess) \
                return kErrUnsupported;                                                                                \
            if (devid >= 0 && devid < 64) attr_done[devid] = true;                                                     \
        }                                                                                                              \
        relax_tail_kernel<PM><<<(unsigned)(point_blocks + pose_blocks), threads, smem, stream>>>(a, point_blocks, Hpad); \
    } while (0)
    if (a.P <= 8) REART_TAIL(8);
    else if (a.P <= 16) REART_TAIL(16);
    else REART_TAIL(32);
#undef REART_TAIL
    REART_CHECK_LAUNCH();
    return kOk;
}

}  // namespace reart
