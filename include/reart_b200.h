/*
 * reart_b200.h -- C ABI of libreart_b200.so: B200 (sm_100a) kernels for reart's per-iteration
 * energy evaluation (skinning -> bidirectional Chamfer nearest-neighbour search -> backward).
 *
 * Conventions (SURVEY.md section 8b; they follow the reference's in-tree native wrappers,
 * networks/pointnet_lib/src/sampling.cpp:11-21, minus the exit(-1)):
 *   - every pointer is DEVICE memory owned by the caller (torch tensors); the library never
 *     allocates or frees; tensors are row-major contiguous; data float32, indices int64;
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it and never
 *     synchronise (except reart_fp32_probe, a benchmark helper);
 *   - return value 0 = success, negative = error (reart_error_string);
 *   - `workspace` is scratch sized by the matching *_workspace_bytes() query, 256-byte aligned.
 *   - reentrant; no global state.
 *
 * Each entry point cites the reference interface (file:line under the reference tree) it replaces.
 */
#ifndef REART_B200_H_
#define REART_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define REART_API __attribute__((visibility("default")))
#else
#define REART_API
#endif

#define REART_OK 0
#define REART_ERR_INVALID_ARG (-1)
#define REART_ERR_WORKSPACE (-2)
#define REART_ERR_LAUNCH (-3)
#define REART_ERR_UNSUPPORTED (-4)

REART_API const char* reart_version(void);
REART_API const char* reart_error_string(int code);
/* the CUDA runtime error behind the most recent REART_ERR_LAUNCH raised by a kernel launch ("none" if there was none) */
REART_API const char* reart_last_cuda_error(void);

/* ---------------------------------------------------------------------------------------------
 * K=1 nearest neighbour, D=3.
 * Replaces chamferdist._C.knn_points_idx(p1, p2, lengths1, lengths2, K=1, version=-1)
 * as called from utils/chamfer.py:174 (via knn_points, utils/chamfer.py:212-286, full lengths).
 *   p1 [B,P1,3], p2 [B,P2,3]  ->  dists [B,P1] squared L2, idx [B,P1] (lowest index on ties).
 * P2 == 0 yields dists = 0, idx = 0 (upstream zero padding).
 * ------------------------------------------------------------------------------------------- */
REART_API int64_t reart_knn1_workspace_bytes(int64_t B, int64_t P1, int64_t P2);
REART_API int reart_knn1_fwd(const float* p1, const float* p2, int64_t B, int64_t P1, int64_t P2, float* dists, int64_t* idx,
                   void* workspace, int64_t workspace_bytes, void* stream);

/* Both directions of ChamferDistance.forward in one pass (utils/chamfer.py:78-94):
 *   src [B,N,3], tgt [B,M,3] -> d_fwd,i_fwd [B,N] (src->tgt) and d_bwd,i_bwd [B,M] (tgt->src). */
REART_API int64_t reart_chamfer_workspace_bytes(int64_t B, int64_t N, int64_t M);
REART_API int reart_chamfer_bidir_fwd(const float* src, const float* tgt, int64_t B, int64_t N, int64_t M, float* d_fwd,
                            int64_t* i_fwd, float* d_bwd, int64_t* i_bwd, void* workspace, int64_t workspace_bytes,
                            void* stream);

/* The search stage of reart_chamfer_bidir_fwd alone (no packing, no index recovery): fills the merge keys
 * keys_a [B,N] / keys_b [B,M] (uint64: dist_bits << 32 | arg-min chunk) from src [B,N,3] and the PACKED tgt.
 * Exposed so benchmarks can time the dominant kernel in isolation; *col_chunk_pts receives the column-chunk
 * width (host pointer, may be NULL); variant 0 = production default; (variant % 16) in 1/2/4/8 = column sub-chunks per warp and
 * (variant / 16) > 0 = forced number of target splits -- tuning knobs only. */
REART_API int reart_chamfer_sym_search(const float* src, const float* tgt_packed, int64_t B, int64_t N, int64_t M,
                                       uint64_t* keys_a, uint64_t* keys_b, int32_t* col_chunk_pts, int variant,
                                       void* stream);

/* ---------------------------------------------------------------------------------------------
 * Backward of the K=1 search.
 * Replaces chamferdist._C.knn_points_backward(p1, p2, lengths1, lengths2, idx, grad_dists)
 * as called from utils/chamfer.py:206-208:
 *   grad_p1[b,i] = 2 g[b,i] (p1[b,i] - p2[b,idx[b,i]]);  grad_p2[b,idx[b,i]] -= same.
 * Both outputs are fully overwritten.
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_knn1_bwd(const float* p1, const float* p2, const int64_t* idx, const float* grad_dists, int64_t B,
                   int64_t P1, int64_t P2, float* grad_p1, float* grad_p2, void* stream);

/* Backward of both directions at once (what autograd sums over the two _knn_points.backward
 * calls, utils/chamfer.py:195-209): g_fwd [B,N], g_bwd [B,M] -> grad_src [B,N,3], grad_tgt [B,M,3].
 * grad_tgt may be NULL (observed frames need no gradient). */
REART_API int reart_chamfer_bidir_bwd(const float* src, const float* tgt, const int64_t* i_fwd, const int64_t* i_bwd,
                            const float* g_fwd, const float* g_bwd, int64_t B, int64_t N, int64_t M, float* grad_src,
                            float* grad_tgt, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Packed cloud layout used by the searches: groups of 4 points [x0..x3|y0..y3|z0..z3], +INF padded to a
 * multiple of 32 points per batch element.  Observed frames are constant over an optimisation, so callers
 * pack them once (reart_pack_cloud) and reuse the buffer every iteration.
 * ------------------------------------------------------------------------------------------- */
REART_API int64_t reart_packed_bytes(int64_t B, int64_t P);
REART_API int reart_pack_cloud(const float* pts, int64_t B, int64_t P, float* packed, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Soft-assignment skinning.
 * Replaces the bmm + broadcast-multiply + sum of networks/model.py:63-69 (BaseModel.forward),
 * networks/model.py:161-165 (KinematicModel.forward) and utils/model_utils.py:54-67 (compute_pc_transform):
 *   out[t,n,:] = sum_p W[n,p] * (R[t,p] @ cano[n] + tr[t,p])
 * cano [N,3], W [N,P] float32, R [T,P,3,3], tr [T,P,3] -> out [T,N,3].
 * Backward: g [T,N,3] -> gW [N,P], gR [T,P,3,3], gtr [T,P,3] (all overwritten).  One pass over g, no atomics:
 * per-chunk pose partials go through the caller's workspace (reart_skin_bwd_workspace_bytes) and are reduced in a
 * fixed order, so the result is bit-identical from run to run.
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_skin_fwd(const float* cano, const float* W, const float* R, const float* tr, int64_t T, int64_t N,
                             int64_t P, float* out, void* stream);
REART_API int64_t reart_skin_bwd_workspace_bytes(int64_t T, int64_t N, int64_t P);
REART_API int reart_skin_bwd(const float* cano, const float* W, const float* R, const float* tr, const float* g,
                             int64_t T, int64_t N, int64_t P, float* gW, float* gR, float* gtr, void* workspace,
                             int64_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * The whole per-iteration energy, fused: skin -> bidirectional Chamfer -> sum -> backward to the
 * skinning inputs.  Equivalent to (networks/model.py:63-69) -> recon_loss (networks/loss.py:24-29,
 * i.e. ChamferDistance(bidirectional=True) utils/chamfer.py:78-123 + torch.sum) -> autograd backward.
 *   cano [N,3], W [N,P], R [T,P,3,3], tr [T,P,3]; tgt [T,M,3] observed frames and their packed copy.
 * Outputs: skinned [T,N,3]; loss[1] (double, sum of all per-point squared distances, both directions);
 *          gW [N,P], gR [T,P,3,3], gtr [T,P,3]; g_skinned [T,N,3] (dLoss/dskinned, may be NULL).
 * compute_grad == 0 stops after the loss.
 * ------------------------------------------------------------------------------------------- */
REART_API int64_t reart_energy_workspace_bytes(int64_t T, int64_t N, int64_t M);
REART_API int reart_skinned_chamfer_fwd_bwd(const float* cano, const float* W, const float* R, const float* tr,
                                            const float* tgt, const float* tgt_packed, int64_t T, int64_t N, int64_t M,
                                            int64_t P, float* skinned, double* loss, float* gW, float* gR, float* gtr,
                                            float* g_skinned, int compute_grad, void* workspace,
                                            int64_t workspace_bytes, void* stream);
/* Same call with the per-point squared distances and arg-min indices of both directions as optional outputs
 * (d_fwd/i_fwd [T,N], d_bwd/i_bwd [T,M]; any may be null): what ChamferDistance(..., return_index=True) of
 * utils/chamfer.py:97-103,119-123 returns, from inside the fused evaluation. */
REART_API int reart_skinned_chamfer_fwd_bwd_ex(const float* cano, const float* W, const float* R, const float* tr,
                                            const float* tgt, const float* tgt_packed, int64_t T, int64_t N, int64_t M,
                                            int64_t P, float* skinned, double* loss, float* gW, float* gR, float* gtr,
                                            float* g_skinned, int compute_grad, float* d_fwd,
                                               int64_t* i_fwd, float* d_bwd, int64_t* i_bwd, void* workspace,
                                            int64_t workspace_bytes, void* stream);
/* The same evaluation with EXACT tile culling (csrc/cull.cu, chamfer_sym.cu: chamfer_sym_cull_kernel): nn_rows [T,N] /
 * nn_cols [T,M] int32 carry the arg-mins from one call to the next (fill with -1 before the first call); together with a
 * history-free coarse descent (clouds of >= 8192 points) they give upper bounds of every minimum, and (256-row, 32-target)
 * blocks whose bounding-box gap is strictly above both bounds are skipped.  Loss, distances, indices and gradients are
 * bit-identical to reart_skinned_chamfer_fwd_bwd_ex for ANY point order and ANY seed values; how much is skipped depends on
 * how spatially compact consecutive points are (engine.py sorts both clouds into a k-d order once).  cull_stats (optional,
 * device, [2] uint64, caller-zeroed): += (warp, chunk) pairs evaluated / offered.  Either nn pointer null: no culling. */
REART_API int reart_skinned_chamfer_fwd_bwd_culled(const float* cano, const float* W, const float* R, const float* tr,
                                                   const float* tgt, const float* tgt_packed, int64_t T, int64_t N,
                                                   int64_t M, int64_t P, float* skinned, double* loss, float* gW,
                                                   float* gR, float* gtr, float* g_skinned, int compute_grad,
                                                   float* d_fwd, int64_t* i_fwd, float* d_bwd, int64_t* i_bwd,
                                                   int32_t* nn_rows, int32_t* nn_cols, uint64_t* cull_stats,
                                                   void* workspace, int64_t workspace_bytes, void* stream);
/* The culled evaluation on the CALLER's point order, bit-identical to reart_skinned_chamfer_fwd_bwd_ex on the same
 * arguments (cano, W, R, tr, tgt in caller order; every output in caller order).  Only the search runs in a permuted order,
 * where consecutive points are spatially compact: row_order [N] (search position -> caller row of cano) with its inverse
 * row_inv, tgt_order [T,M] (per frame: search position -> caller target) with tgt_inv; tgt_search [T,M,3] = tgt in
 * tgt_order, tgt_search_packed its reart_pack_cloud copy.  Culling is exact for any order, and index ties are exact: the
 * search marks every point whose minimum is reached in two of its chunks, and those take the lowest caller index among
 * all points at exactly that distance -- the brute force's answer.  Points ordered by caller index inside every 256-row
 * block and 32-target chunk of the search order are required for the others: a chunk's first match is then its lowest
 * caller index.  nn_rows [T,N] / nn_cols [T,M] (device, int32, by CALLER index: nn_rows[t][i] the arg-min caller target
 * of caller row i, nn_cols[t][j] the arg-min caller row of caller target j) are the culling seeds as in
 * reart_skinned_chamfer_fwd_bwd_culled (-1 / any value: still exact) and are overwritten with this evaluation's arg-mins;
 * they do not depend on the search order, so they carry over when the order changes.
 * stats (optional, device, [3] uint64, caller-zeroed): += (warp, chunk) pairs evaluated, offered, points resolved by the
 * tie path. */
REART_API int reart_skinned_chamfer_fwd_bwd_ordered(const float* cano, const float* W, const float* R, const float* tr,
                                                    const float* tgt, const float* tgt_search, const float* tgt_search_packed,
                                                    int64_t T, int64_t N, int64_t M, int64_t P, const int32_t* row_order,
                                                    const int32_t* row_inv, const int32_t* tgt_order, const int32_t* tgt_inv,
                                                    float* skinned, double* loss, float* gW, float* gR, float* gtr,
                                                    float* g_skinned, int compute_grad, float* d_fwd, int64_t* i_fwd,
                                                    float* d_bwd, int64_t* i_bwd, int32_t* nn_rows, int32_t* nn_cols,
                                                    uint64_t* stats, void* workspace, int64_t workspace_bytes, void* stream);
/* reart_skinned_chamfer_fwd_bwd_ordered with a row order the call computes itself, per frame, on the skinned cloud
 * (csrc/order.cu): a sort-tile-recursive order -- the frame's axes by decreasing extent; rows sorted by (coordinate, caller
 * index) along the first into slabs of 2048, each slab along the second into pieces of 512, each piece along the third into
 * leaves of 256 (the last leaf of a frame may be short); every leaf then in ascending caller index.  Once the parts of a fit
 * move apart, the skinned rows of one canonical neighbourhood land in many places of a frame, and blocks grouped on the
 * posed cloud stay compact where a fixed order does not.  row_order / row_inv [T,N] (device, int32) are written: search
 * position -> caller row and its inverse.  Every other argument and result as in reart_skinned_chamfer_fwd_bwd_ordered;
 * bit-identical to reart_skinned_chamfer_fwd_bwd_ex.  N <= reart_posed_order_max_points() (else REART_ERR_UNSUPPORTED). */
REART_API int reart_skinned_chamfer_fwd_bwd_posed(const float* cano, const float* W, const float* R, const float* tr,
                                                  const float* tgt, const float* tgt_search, const float* tgt_search_packed,
                                                  int64_t T, int64_t N, int64_t M, int64_t P, const int32_t* tgt_order,
                                                  const int32_t* tgt_inv, int32_t* row_order, int32_t* row_inv,
                                                  float* skinned, double* loss, float* gW, float* gR, float* gtr,
                                                  float* g_skinned, int compute_grad, float* d_fwd, int64_t* i_fwd,
                                                  float* d_bwd, int64_t* i_bwd, int32_t* nn_rows, int32_t* nn_cols,
                                                  uint64_t* stats, void* workspace, int64_t workspace_bytes, void* stream);
REART_API int64_t reart_posed_order_max_points(void);
/* The same energy with the skinning FUSED INTO THE PRODUCER SIDE OF THE SEARCH (the composition networks/model.py:63-69 ->
 * utils/chamfer.py:78-94 in one kernel): every search CTA skins its own 2048 canonical points in its prologue and the
 * skinned cloud / x-sorted copy are emitted as by-products, so there is no skinning launch and the cloud is not re-read.
 * For one-hot weight rows (what F.gumbel_softmax(hard=True) and one_hot give, networks/model.py:44,150): hot [N,2] is the
 * compact form (part id as int32 bits, weight value) written by reart_relax_head; W [N,P] is still read by the backward.
 * Results are bit-identical to reart_skinned_chamfer_fwd_bwd.  cano, hot, skinned 16-byte aligned. */
REART_API int reart_skinned_chamfer_fwd_bwd_fused(const float* cano, const float* hot, const float* W, const float* R,
                                                  const float* tr, const float* tgt, const float* tgt_packed, int64_t T,
                                                  int64_t N, int64_t M, int64_t P, float* skinned, double* loss, float* gW,
                                                  float* gR, float* gtr, float* g_skinned, int compute_grad,
                                                  void* workspace, int64_t workspace_bytes, void* stream);


/* ---------------------------------------------------------------------------------------------
 * Segmentation head and straight-through gumbel weights (the per-point, frame-independent part of an iteration).
 * reart_segmlp_fwd/bwd replace MLPConv1d(3,(H,P)) = Conv1d(3,H,1,bias)+ReLU+Conv1d(H,P,1,no bias)
 * (networks/blocks.py:99-118, built at networks/model.py:19, applied at :42-43): x [N,3], w0 [H,3], b0 [H],
 * w2 [P,H] -> logits [N,P]; backward: glogits [N,P] -> gw0 [H,3], gb0 [H], gw2 [P,H] (overwritten).
 * reart_gumbel_st_fwd/bwd replace F.gumbel_softmax(logits, tau, hard=True) (networks/model.py:44) given
 * expo [N,P] ~ Exponential(1) drawn by torch and tau[1] on the device: -> W [N,P] (straight-through weights) and
 * ysoft [N,P] (saved); backward: gW [N,P] -> glogits [N,P].   H <= 1024, P <= 32.
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_segmlp_fwd(const float* x, const float* w0, const float* b0, const float* w2, int64_t N, int64_t H,
                               int64_t P, float* logits, void* stream);
REART_API int reart_segmlp_bwd(const float* x, const float* w0, const float* b0, const float* w2, const float* glogits,
                               int64_t N, int64_t H, int64_t P, float* gw0, float* gb0, float* gw2, void* stream);
REART_API int reart_gumbel_st_fwd(const float* logits, const float* expo, const float* tau, int64_t N, int64_t P,
                                  float* W, float* ysoft, void* stream);
REART_API int reart_gumbel_st_bwd(const float* ysoft, const float* tau, const float* gW, int64_t N, int64_t P,
                                  float* glogits, void* stream);

/* ---------------------------------------------------------------------------------------------
 * The frame-independent part of one relaxation iteration (run_robot.py:154-221, --model=base), fused.
 * head: seg MLP forward (networks/blocks.py:99-118 via networks/model.py:42-43) + straight-through gumbel-softmax
 *       weights from caller-drawn Exponential(1) noise `expo` (F.gumbel_softmax(hard=True), networks/model.py:44)
 *       + 6D -> R (networks/model.py:60).  cano [N,3]; w0 [H,3], b0 [H], w2 [P,H]; expo [N,P]; tau [1]; d6 [T,P,6]
 *       -> logits [N,P] (optional), W [N,P], ysoft [N,P], R [T,P,3,3].  noise_index [N] (optional): point n uses noise row
 *       noise_index[n] -- for callers that reordered the cloud but want the random decisions of the original order.
 *       hot [N,2] (optional, 16-byte aligned): every row of W has exactly one non-zero; (its part as int32 bits, its value)
 *       is written here for reart_skinned_chamfer_fwd_bwd_fused.
 * tail: gumbel backward + seg MLP backward + 6D backward + (frames sharded over `world` ranks: the one-shot
 *       peer-memory all-reduce of reart_allreduce_oneshot, inline) + Adam with torch.optim.Adam semantics
 *       (run_robot.py:146-150, 219-221) on w0/b0/w2 (lr_seg) and d6/tr (lr_pose), all in ONE launch with a fixed
 *       summation order (bit-reproducible).  `tickets` [reart_relax_tail_ticket_words(N)] uint32 must be zero before the
 *       first call only (the kernel re-arms them).
 *       phase 0: everything; phase 1: gradients -> bucket only (caller reduces the bucket, e.g. with NCCL);
 *       phase 2: Adam from the reduced bucket.
 * limits: P <= 32 for both.  The head stages w0/b0/w2 in shared memory and rejects H*(8+PMAX)*4 > 48 KB with
 *       REART_ERR_UNSUPPORTED, PMAX being P rounded up to 8, 16 or 32 (e.g. P > 16 with H > 307 is unsupported).  The tail
 *       supports H <= 256 (REART_ERR_UNSUPPORTED above that).
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_relax_head(const float* cano, const float* w0, const float* b0, const float* w2, const float* expo,
                               const int64_t* noise_index, const float* tau, const float* d6, int64_t N, int64_t H, int64_t P, int64_t T,
                               float* logits, float* W, float* ysoft, float* R, float* hot, void* stream);
typedef struct reart_relax_tail_args {
    const float* cano;
    float* w0; float* b0; float* w2;
    const float* ysoft; const float* tau; const float* gW;
    float* d6; float* tr;
    const float* gR; const float* gtr;
    float* m_seg; float* v_seg; float* m_d6; float* v_d6; float* m_tr; float* v_tr;
    float* step;
    float lr_pose, lr_seg, beta1, beta2, eps, weight_decay;
    float* partials;              /* reart_relax_tail_workspace_bytes(N,H,P) */
    uint32_t* tickets;
    const double* loss_local;
    float* bucket;                /* [4H + PH + 1] */
    float* loss_out;
    const uint64_t* peer_base; uint32_t* epoch; int32_t rank, world, n_pad;
    int32_t phase;
    int64_t N, H, P, T;
} reart_relax_tail_args;
REART_API int64_t reart_relax_tail_workspace_bytes(int64_t N, int64_t H, int64_t P);
REART_API int64_t reart_relax_tail_ticket_words(int64_t N);
REART_API int reart_relax_tail(const reart_relax_tail_args* args, void* stream);

/* ---------------------------------------------------------------------------------------------
 * One iteration of the kinematic (projection) model (run_robot.py's second model, --model=kinematic), fused around the
 * energy (reart_skinned_chamfer_fwd_bwd / _ordered with the constant one-hot weights of the label transfer).
 * head: KinematicModel.transforms (networks/model.py:151-159): tree forward kinematics of reart_fk_fwd
 *       (utils/kinematic_utils.py:151-198, same tree arrays, same device arithmetic) followed by the optional learned
 *       root pose root @ fk, root = [rotation_6d_to_matrix(root_6d) | root_t] (networks/model.py:155-158).
 *       axis, moment [E,3], theta [T,E], distance [T,E] or NULL, joint_type [E] or NULL; root_6d [T,6] and root_t [T,3]
 *       both or neither -> R [T,P,3,3], tr [T,P,3] (the energy's pose inputs; without a root pose bit-identical to
 *       reart_fk_fwd's [..., :3, :3] / [..., :3, 3]) and fk [T,P,12] (the 3x4 poses before the root pose, for the tail).
 * tail: the backward of head given d loss / d (R, tr) from the energy (dual-number screw derivatives, frame sums in frame
 *       order -- no float atomics, bit-reproducible), [frames sharded over `world` ranks: the one-shot peer-memory
 *       all-reduce of reart_allreduce_oneshot, inline, on grad[0 .. 6E]] and Adam with torch.optim.Adam semantics and one
 *       learning rate (run_robot.py:146-150, 219-221 as the kinematic run builds it) on every parameter, in ONE launch.
 *       grad (written) = [g_axis 3E | g_moment 3E | loss | g_theta T*E | g_distance T*E (with distance) | g_root_6d 6T,
 *       g_root_t 3T (with a root pose)]; m, v: Adam moments in the same layout; step [1] counts completed steps.
 *       phase 0: everything; 1: gradients only (the caller reduces grad[0 .. 6E], e.g. with NCCL); 2: Adam from grad.
 * P <= 32; joint_type values as in reart_fk_fwd.  A one-part model (P = 1) has no joints: axis, moment and theta may be
 * NULL in both calls, and only the root pose (if any) trains.
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_kin_head(const float* axis, const float* moment, const float* theta, const float* distance,
                             const int32_t* order, const int32_t* parent, const int32_t* edge, const int32_t* joint_type,
                             const float* root_6d, const float* root_t, int64_t T, int64_t P, float* R, float* tr, float* fk,
                             void* stream);
typedef struct reart_kin_tail_args {
    const float* fk;
    const float* gR; const float* gtr;
    const double* loss_local;
    const int32_t* order; const int32_t* parent; const int32_t* edge; const int32_t* joint_type;
    float* axis; float* moment; float* theta; float* distance; float* root_6d; float* root_t;
    float* grad; float* m; float* v;
    float* step;
    float lr, beta1, beta2, eps, weight_decay;
    float* partials;              /* reart_kin_tail_workspace_bytes(T,P) */
    float* loss_out;
    const uint64_t* peer_base; uint32_t* epoch; int32_t rank, world, n_pad;
    int32_t phase;
    int64_t T, P;
} reart_kin_tail_args;
REART_API int64_t reart_kin_tail_workspace_bytes(int64_t T, int64_t P);
REART_API int reart_kin_tail(const reart_kin_tail_args* args, void* stream);

/* The assignment loss of the kinematic model (run_robot.py:181-187) straight into the pose gradients, between the energy
 * (or reart_skin_fwd) and reart_kin_tail.  Premise: the skinning weights are ONE-HOT rows (the kinematic model's label
 * transfer), so the gradient w.r.t. (R, tr) of part p in frame t is a sum over the samples of part p alone:
 *   d = skinned[t, src_idx[i]] - tgt[t, col4row[t,i]],  x = cano[src_idx[i]]
 *   loss += lambda sum |d|^2,  gR[t,p] += 2 lambda sum d x^T,  gtr[t,p] += 2 lambda sum d.
 * skinned [T,N,3] (read, not recomputed), cano [N,3], src_idx [n] int64, tgt [T,n,3] (the sampled targets), col4row [T,n]
 * (reart_lap); sample_order [n]: the sample indices stably sorted by the part of cano[src_idx[i]], part_offsets [P+1]: part
 * p owns sample_order[part_offsets[p] .. part_offsets[p+1]).  gR [T,P,3,3], gtr [T,P,3], loss [1] double: accumulate != 0
 * adds to them (after the energy wrote its Chamfer gradients), else overwrites them (a part without samples gets zeros;
 * with accumulate its gradient is left untouched).  No float atomics: bit-reproducible.  workspace:
 * reart_kin_assign_workspace_bytes(T,P), zero before the FIRST call (the kernel re-arms it).  P <= 32, n <= 4096 as reart_lap.
 * ------------------------------------------------------------------------------------------- */
REART_API int64_t reart_kin_assign_workspace_bytes(int64_t T, int64_t P);
REART_API int reart_kin_assign(const float* skinned, const float* cano, const int64_t* src_idx, const float* tgt,
                               const int32_t* col4row, const int32_t* sample_order, const int32_t* part_offsets,
                               float lambda, int64_t T, int64_t N, int64_t n, int64_t P, float* gR, float* gtr,
                               double* loss, int accumulate, void* workspace, int64_t workspace_bytes, void* stream);

/* The flow loss of the kinematic model (run_robot.py:194-213, networks/loss.py:10-21) straight into the pose gradients,
 * between the energy (or reart_skin_fwd) and reart_kin_tail.  Same premise as reart_kin_assign: one-hot skinning weights,
 * so the gradient w.r.t. (R, tr) of part p in frame t is a sum over the points of part p.  The kernel works on a WINDOW
 * of the complete sequence (canonical cloud inserted at cano_idx): win [K,N,3] holds K consecutive complete frames,
 * tflow [K-1,N,3] / mask [K-1,N] (uint8, as reart_knn3_blend writes them) the blended target flow of pair k = (slot k,
 * slot k+1), slot_frame [K] int32 the local frame of each slot (-1: the canonical cloud or a neighbour rank's frame).
 *   pred_k = win[k+1] - win[k],  err_k = pred_k - tflow[k],  per point and component d_k = d flow_loss / d pred_k:
 *     mask set, plain: 2 err;  mask set, robust: err where |err| < 1, else sign(err) (|err| == 1 takes the linear branch,
 *     as torch.where(a < 1, ...) does);  mask clear: 2 * 0.01 * pred.
 *   slot s holding local frame t, point i of part p, x = cano[i]:  g = lambda (d_{s-1} - d_s) (a pair outside the window
 *   is dropped);  gR[t,p] += sum g x^T,  gtr[t,p] += sum g.
 *   loss += lambda * sum over the pairs [q0, q1) of the window of the per-point terms (mask set: |err|^2, or the Huber
 *   terms 0.5 e^2 / |e| - 0.5 when robust; mask clear: 0.01 |pred|^2).  Pair k is counted by slot k+1 when that slot
 *   is local, else by slot k (a counted pair needs a local slot).
 * A frame's gradient depends only on its own slot and the two adjacent ones: a sub-window that holds a frame's
 * neighbours gives that frame the bits of the whole-sequence call.  point_order [N]: the point indices stably sorted by
 * part, part_offsets [P+1]: part p owns point_order[part_offsets[p] .. part_offsets[p+1]).  gR [T,P,3,3], gtr [T,P,3],
 * loss [1] double: accumulate != 0 adds to them, else overwrites them (every local frame's (t, p) is written; a part
 * without points gets zeros, with accumulate it is left untouched).  No float atomics: bit-reproducible.  workspace:
 * reart_kin_flow_workspace_bytes(K,P), zero before the FIRST call (the kernel re-arms it).  P <= 32, K >= 2,
 * 0 <= q0 <= q1 <= K-1; T == 0 is an empty problem.
 * ------------------------------------------------------------------------------------------- */
REART_API int64_t reart_kin_flow_workspace_bytes(int64_t K, int64_t P);
REART_API int reart_kin_flow(const float* win, const float* tflow, const uint8_t* mask, const int32_t* slot_frame,
                             const float* cano, const int32_t* point_order, const int32_t* part_offsets, float lambda,
                             int robust, int64_t K, int64_t N, int64_t P, int64_t T, int64_t q0, int64_t q1, float* gR,
                             float* gtr, double* loss, int accumulate, void* workspace, int64_t workspace_bytes,
                             void* stream);

/* The flow loss (run_robot.py:194-213, networks/loss.py:10-21) and its gradient w.r.t. the SKINNED cloud, for a model
 * whose skinning weights train (the relaxation model: reart_skin_bwd takes the gradient on to gW, gR, gtr).  Between the
 * energy (compute_grad = 0, g_skinned set) or reart_skin_fwd and reart_skin_bwd.  Same window as reart_kin_flow: win [K,N,3]
 * holds K consecutive frames of the complete sequence (canonical cloud inserted at cano_idx), tflow [K-1,N,3] / mask [K-1,N]
 * (uint8, as reart_knn3_blend writes them) the blended target flow of pair k = (slot k, slot k+1), slot_frame [K] int32 the
 * local frame of each slot (-1: the canonical cloud or a neighbour rank's frame).
 *   pred_k = win[k+1] - win[k],  err_k = pred_k - tflow[k],  per point and component d_k = d flow_loss / d pred_k:
 *     mask set, plain: 2 err;  mask set, robust: err where |err| < 1, else sign(err) (|err| == 1 takes the linear branch);
 *     mask clear: 2 * 0.01 * pred   (the per-component rule of reart_kin_flow, the same operations).
 *   slot s holding local frame t, point i, component r:  g_skinned[t,i,r] (+)= lambda (d_{s-1} - d_s)  (a pair outside the
 *   window is dropped).
 *   loss += lambda * sum over the pairs [q0, q1) of the window of the per-point terms, each pair counted by slot k+1 when
 *   that slot is local, else by slot k, exactly as reart_kin_flow counts it.
 * A frame's gradient depends only on its own slot and the two adjacent ones: a sub-window that holds a frame's neighbours
 * gives that frame the bits of the whole-sequence call.  g_skinned [T,N,3] in the caller's point order, loss [1] double:
 * accumulate != 0 adds to them (one float add per element), else overwrites them (every point of every local frame that
 * has a slot is written, the loss slot is set).  No float atomics: bit-reproducible.  workspace:
 * reart_flow_grad_workspace_bytes(K,N), zero before the FIRST call (the kernel re-arms it).  K >= 2, N >= 1,
 * 0 <= q0 <= q1 <= K-1; T == 0 is an empty problem.
 * ------------------------------------------------------------------------------------------- */
REART_API int64_t reart_flow_grad_workspace_bytes(int64_t K, int64_t N);
REART_API int reart_flow_grad(const float* win, const float* tflow, const uint8_t* mask, const int32_t* slot_frame,
                              float lambda, int robust, int64_t K, int64_t N, int64_t T, int64_t q0, int64_t q1,
                              float* g_skinned, double* loss, int accumulate, void* workspace, int64_t workspace_bytes,
                              void* stream);

/* ---------------------------------------------------------------------------------------------
 * 6D rotation representation -> matrix (Gram-Schmidt).
 * Replaces screw_se3/geo_utils.py:632-651 (rotation_6d_to_matrix); d6 [B,6] -> R [B,3,3].
 * Backward: gR [B,3,3] -> gd6 [B,6].
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_rot6d_fwd(const float* d6, int64_t B, float* R, void* stream);
REART_API int reart_rot6d_bwd(const float* d6, const float* gR, int64_t B, float* gd6, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Screw parameters -> 4x4 transform.
 * Replaces transform_from_exponential_coordinates(screw_param_to_exponential_coordinates(l, m, theta, d))
 * (screw_se3/screw_utils.py:6-30 over se3_exp_map, screw_se3/geo_utils.py:147-222), quirks included.
 *   l,m [B,3], theta,d [B] -> M [B,4,4].   Backward: gM [B,4,4] -> gl, gm [B,3], gtheta, gd [B].
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_screw_to_transform_fwd(const float* l, const float* m, const float* theta, const float* d,
                                           int64_t B, float* M, void* stream);
REART_API int reart_screw_to_transform_bwd(const float* l, const float* m, const float* theta, const float* d,
                                           const float* gM, int64_t B, float* gl, float* gm, float* gtheta, float* gd,
                                           void* stream);

/* ---------------------------------------------------------------------------------------------
 * Forward kinematics over the joint tree.
 * Replaces fk(paths_to_base, reverse_topo, edge_index, axis_list, moment_list, theta_list,
 *             distance_list, joint_type_list)  (utils/kinematic_utils.py:151-198).
 * The dict-based tree is passed flattened (device int32 arrays): order[P] = reverse_topo (root first),
 * parent[P] (-1 for the root), edge[P] = index of the edge joining a part to its parent,
 * joint_type[E] (0 as given / 1 revolute / 2 prismatic) or NULL; distance [T,E] or NULL (d = 1e-6).
 *   axis, moment [E,3], theta [T,E] -> out [T,P,4,4] indexed by part id.
 * Backward: g_out [T,P,4,4] -> g_axis, g_moment [E,3], g_theta [T,E], g_dist [T,E] (NULL if distance NULL);
 * workspace: T*P*16 floats.
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_fk_fwd(const float* axis, const float* moment, const float* theta, const float* distance,
                           const int32_t* order, const int32_t* parent, const int32_t* edge, const int32_t* joint_type,
                           int64_t T, int64_t P, float* out, void* stream);
REART_API int reart_fk_bwd(const float* axis, const float* moment, const float* theta, const float* distance,
                           const int32_t* order, const int32_t* parent, const int32_t* edge, const int32_t* joint_type,
                           int64_t T, int64_t P, const float* fk_out, const float* g_out, float* g_axis,
                           float* g_moment, float* g_theta, float* g_dist, float* workspace, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Small-k nearest neighbours with EUCLIDEAN distances, ascending, ties -> lowest index.
 * Replaces knn_cuda.KNN(k, transpose_mode=True)(ref, query) (KNN_CUDA 0.2; call sites
 * utils/flow_utils.py:158, utils/model_utils.py:42):  ref [B,n,3], query [B,m,3] -> dist, idx [B,m,k], k <= 8.
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_knn(const float* ref, const float* query, int64_t B, int64_t n, int64_t m, int k, float* dist,
                        int64_t* idx, void* stream);
/* The same search returning SQUARED distances (the chamferdist._C.knn_points_idx contract for K > 1,
 * utils/chamfer.py:174-189; the reference itself only ever uses K == 1). */
REART_API int reart_knn_sq(const float* ref, const float* query, int64_t B, int64_t n, int64_t m, int k, float* dist,
                           int64_t* idx, void* stream);

/* Flow blending for all frame pairs at once.  Replaces the Python loop over
 * blend_anchor_motion(query, ref, flow, knn_flow, return_mask=True) (utils/flow_utils.py:147-170,
 * called T times per iteration from run_robot.py:199-202) with k = 3.
 *   query [T,m,3]; ref_cat/flow_cat [sum n_t,3] (the per-pair lists concatenated);
 *   ref_offsets [T+1] int64 DEVICE array of row offsets -> blended [T,m,3], mask [T,m] (uint8 0/1). */
REART_API int reart_knn3_blend(const float* query, const float* ref_cat, const float* flow_cat,
                               const int64_t* ref_offsets, int64_t T, int64_t m, float* blended, uint8_t* mask,
                               void* stream);

/* The same blend, bit-identical results, for reference sets that stay fixed over many calls (they do: run_robot.py:78-84
 * builds pc_ref_list / flow_ref_list once, the loop of :199-202 queries them every iteration).
 *   reart_flow_refs_sort: once per fit -- sorts every pair's references along x into `sorted`
 *     (reart_flow_refs_sorted_bytes(total_refs, T) bytes) and writes each pair's start (in 64-byte groups) to
 *     sorted_offsets [T] int64 (device).  max_refs = the largest per-pair count (host value, <= 16384, else
 *     REART_ERR_UNSUPPORTED: use reart_knn3_blend).
 *   reart_knn3_blend_sorted: per call -- buckets the queries by x (query_order [T,m] int32 scratch) and searches only
 *     the x-slab of references that can still hold one of the 3 nearest (exact: a skipped reference has
 *     dx*dx > current 3rd best; ties by lowest original index as in reart_knn3_blend). */
REART_API int64_t reart_flow_refs_sorted_bytes(int64_t total_refs, int64_t T);
REART_API int reart_flow_refs_sort(const float* ref_cat, const int64_t* ref_offsets, int64_t T, int64_t max_refs,
                                   void* sorted, int64_t sorted_bytes, int64_t total_refs, int64_t* sorted_offsets,
                                   void* stream);
REART_API int reart_knn3_blend_sorted(const float* query, const void* sorted, const int64_t* sorted_offsets,
                                      const float* flow_cat, const int64_t* ref_offsets, int64_t T, int64_t m,
                                      int32_t* query_order, float* blended, uint8_t* mask, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Assignment loss (run_robot.py:164-187, run_real.py:180-203, run_sapien.py:179-203; utils/model_utils.py:85-103).
 * reart_lap: for each of B frames the exactly optimal one-to-one matching of n source samples to n target samples
 *   under the float32 Euclidean cost (what linear_sum_assignment(torch.cdist(pc_src, pc_tgt)) returns on the host in
 *   the reference), by shortest augmenting paths with float64 duals, costs formed on the fly -- no n x n matrix, no
 *   D2H copy, no host solver.  Source sample i of frame b is src[b][src_idx[i]] (src_idx may be null: i itself);
 *   src has src_points points per frame.  col4row [B,n] int32: target sample matched to source sample i (rows in
 *   order, like scipy's row_ind = arange).  total [B] float64 (optional): the assignment's cost.  n <= 4096.
 *   dual_u [B,n] float64 (optional): the row duals of the solve are written there; with warm_start != 0 they are also
 *   READ as the starting duals (a previous solve of slightly different clouds -- the refresh every assign_gap
 *   iterations): any starting duals give the same optimal cost, good ones leave almost no augmentation to do.
 * reart_assign_loss_grad: loss += lambda * sum |skinned[t, src_idx[i]] - tgt[t, col4row[t,i]]|^2 and its gradient
 *   into g_skinned [T,N,3] (accumulate != 0: added to what is there; else written at the sampled points only).
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_lap(const float* src, const int64_t* src_idx, int64_t src_points, const float* tgt, int64_t B,
                        int64_t n, int32_t* col4row, double* total, double* dual_u, int warm_start, void* stream);
REART_API int reart_assign_loss_grad(const float* skinned, const int64_t* src_idx, const float* tgt,
                                     const int32_t* col4row, int64_t T, int64_t N, int64_t n, float lambda,
                                     float* g_skinned, int accumulate, double* loss, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Furthest point sampling / ball query (the two reachable kernels of the reference's PointNet++ extension).
 * Replace pointnet2_cuda.furthest_point_sampling_wrapper(B, N, npoint, xyz, temp, out) and
 * pointnet2_cuda.ball_query_wrapper(B, N, npoint, radius, nsample, new_xyz, xyz, idx)
 * (networks/pointnet_lib/pointnet2_utils.py:29,263; kernels networks/pointnet_lib/src/sampling_gpu.cu:93-209,
 * ball_query_gpu.cu:9-45).  FPS starts at index 0; arg-max ties -> lowest index.  N <= 32768 per cloud.
 *   xyz [B,N,3] -> out [B,npoint] int32;   new_xyz [B,m,3], xyz [B,N,3] -> idx [B,m,nsample] int32
 *   (idx must be zero-filled by the caller, as the reference does).
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_fps(const float* xyz, int64_t B, int64_t N, int64_t npoint, int32_t* out, void* stream);
/* The wrapper's full signature (furthest_point_sampling_wrapper(B, N, npoint, xyz, temp, out),
 * networks/pointnet_lib/pointnet2_utils.py:29): temp [B,N] float32 scratch lifts the N <= 32768 limit of reart_fps
 * (clouds up to that size ignore it).  Same samples as reart_fps. */
REART_API int reart_fps_temp(const float* xyz, int64_t B, int64_t N, int64_t npoint, float* temp, int32_t* out,
                             void* stream);
REART_API int reart_ball_query(const float* new_xyz, const float* xyz, int64_t B, int64_t N, int64_t m, float radius,
                               int nsample, int32_t* idx, void* stream);

/* ---------------------------------------------------------------------------------------------
 * One-shot all-reduce (sum, in place) of a small float bucket over NVLink peer memory -- the single collective of
 * the frame-sharded iteration (SURVEY.md section 8e; the reference has no distributed code).
 *   peer_base [world] (DEVICE array of uint64): base address of every rank's symmetric, peer-mapped allocation of
 *     (2*n_pad floats + world uint32) zero-initialised bytes (e.g. torch.distributed._symmetric_memory);
 *   epoch [1] uint32 on this device, zero-initialised, owned by this communicator; data [n] floats, n <= n_pad.
 * Every rank must call it the same number of times; all ranks receive bitwise identical sums.
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_allreduce_oneshot(const uint64_t* peer_base, int rank, int world, int64_t n, int64_t n_pad,
                                      uint32_t* epoch, float* data, void* stream);

/* ---------------------------------------------------------------------------------------------
 * FP32-pipe micro-benchmark (roofline denominator; BASELINE.md section 3).  Runs variant
 * 0..5 (see csrc/probe.cu) once warm and once timed with CUDA events on `stream`, SYNCHRONISES,
 * and returns milliseconds and the number of measured lane-operations per thread.
 * scratch_in: >= 1024 floats (any finite values), scratch_out: >= blocks*256 floats.
 * ------------------------------------------------------------------------------------------- */
REART_API int reart_fp32_probe(int variant, int iters, int blocks, const float* scratch_in, float* scratch_out, double* ms,
                     double* ops_per_thread, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* REART_B200_H_ */
