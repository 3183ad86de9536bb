// kernels.h -- internal launcher interface between the .cu translation units and capi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace reart {

// One search direction: every query of `q` against the packed targets `tpacked`.
struct KnnDir {
    const float* q;               // [B, nq, 3] queries (AoS)
    const float* tpacked;         // [B, nt_pad/4, 12] packed targets (common.cuh layout)
    unsigned long long* keys;     // [B, nq] (dist_bits << 32 | chunk) merge keys
    float* out_dists;             // [B, nq] or null   (finalize)
    int64_t* out_idx;             // [B, nq] or null   (finalize)
    int nq;                       // queries per batch element
    int nt;                       // real targets per batch element
    int nt_pad;                   // padded targets (multiple of kChunk)
    int qblocks;                  // filled by the launcher
    int splits;                   // filled by the launcher
    int keys_preset;              // 1: caller already set keys to 0xff.. (fused pipelines)
    int chunk_pts;                // targets per arg-min chunk recorded in the key (finalize re-scan span)
    const unsigned char* perm;    // null, or [B,nt_pad]: tpacked is x-sorted per chunk_pts block (perm = original offset)
    const float* xq;              // with perm: [B, nt_pad/256, 16] quantile index of every sorted block (common.cuh)
};

struct KnnParams {
    KnnDir dir[2];
    int ndir;
    int B;
    int items0;                   // number of work items of dir[0]
};

// Symmetric bidirectional search (chamfer_sym.cu): A rows in registers, B columns streamed.
struct SymParams {
    const float* a;               // [B, na, 3]
    const float* b_packed;        // [B, nb_pad/4, 12]
    unsigned long long* keys_a;   // [B, na]  row keys   (chunk = 32 B-points)
    unsigned long long* keys_b;   // [B, nb]  column keys (chunk = col_chunk_pts A-points)
    int B, na, nb, nb_pad;
    int qblocks, splits;          // filled by the launcher
    int col_chunk_pts;            // filled by the launcher (32 * R / S)
    int keys_preset;
    int keys_one_allocation;      // 1: keys_a and keys_b are carved from one workspace (a single memset may span both)
    int variant;                  // 0 = default; 1/2/4/8 = number of column sub-chunks per warp (tuning)
    unsigned* col_bound;          // null, or one word (zero on entry): atomicMax of the finite column minima every CTA
                                  // saw, as float bits -- an upper bound of every final column minimum (energy.cu)
    // exact tile culling (cull.cu builds these; chamfer_sym.cu CULL = true consumes them)
    int cull;                     // 1: use the culled schedule
    const float* colbox;          // [B, nb_pad/32, 8]: lo.xyz, hi.xyz of the chunk's real points, upper bound of its columns' minima, pad
    const float* rowbound;        // [B, ceil(na/256)]: upper bound of the final minima of each 256-row chunk
    int row_chunks;               // filled by the launcher
    unsigned long long* cull_stats;   // null, or [2] (zero on entry): (warp, chunk) pairs evaluated / offered
    unsigned* tie_a;              // null, or [B,na] followed by tie_b [B,nb]: tie words of the culled search (chamfer_sym.cu
    unsigned* tie_b;              // TIES), set to 0xffffffff by the launcher
    // fused producer (chamfer_sym.cu SKIN = true): sk_cano != null -> `a` is not read, the rows are skinned in the kernel
    const float* sk_cano;         // [na,3] canonical cloud
    const float* sk_hot;          // [na,2] one-hot weights in compact form: (part as int bits, weight value)
    const float* sk_R;            // [B,P,9]
    const float* sk_tr;           // [B,P,3]
    int sk_P, sk_npad;            // parts; padded points of the sorted copy (multiple of 256)
    float* sk_out;                // out [B,na,3] skinned cloud (AoS)
    float* sk_sorted;             // out [B,sk_npad*3] x-sorted blocks (common.cuh layout)
    unsigned char* sk_perm;       // out [B,sk_npad]
    float* sk_xq;                 // out [B,sk_npad/256,16]
};
struct CullParams {
    const float* a;               // [B,na,3] rows (skinned cloud)
    const float* b;               // [B,nb,3] columns (observed frames)
    // seeds from an EARLIER evaluation, by caller index (-1: unknown): nn_rows [B,na] the arg-min caller target of every
    // caller row, nn_cols [B,nb] the arg-min caller row of every caller target
    const int32_t* nn_rows;
    const int32_t* nn_cols;
    // a, b in a search order (null: caller order): row_order / row_inv [row_stride ? B : 1, na] (search position <-> caller
    // row; row_stride 0: one order for all frames, na: one per frame), tgt_order / tgt_inv [B,nb]
    const int32_t* row_order; const int32_t* row_inv; const int32_t* tgt_order; const int32_t* tgt_inv;
    int64_t row_stride;
    int B, na, nb, nb_pad;
    float* colbox;                // out [B, nb_pad/32, 8]
    float* rowbound;              // out [B, ceil(na/256)]
    int coarse;                   // 1: also bound every point by a history-free coarse descent over the other cloud (cull.cu)
};
int launch_cull_bounds(const CullParams& p, cudaStream_t stream);

int launch_pack_cloud(const float* pts, float* packed, int64_t B, int64_t P, cudaStream_t stream);
int launch_pack_cloud_sorted(const float* pts, float* packed, unsigned char* perm, float* xq, int64_t B, int64_t P,
                             int64_t n_pad, cudaStream_t stream);
int launch_knn1_search(KnnParams& p, cudaStream_t stream);
int launch_knn1_finalize(const KnnParams& p, cudaStream_t stream);
int launch_chamfer_sym(SymParams& p, cudaStream_t stream);

int launch_knn1_bwd(const float* p1, const float* p2, const int64_t* idx, const float* grad_dists, int64_t B,
                    int64_t P1, int64_t P2, float* grad_p1, float* grad_p2, int accumulate, cudaStream_t stream);

int launch_chamfer_bidir_bwd(const float* src, const float* tgt, const int64_t* i_fwd, const int64_t* i_bwd,
                             const float* g_fwd, const float* g_bwd, int64_t B, int64_t N, int64_t M, float* grad_src,
                             float* grad_tgt, cudaStream_t stream);

int launch_skin_fwd(const float* cano, const float* W, const float* R, const float* tr, int64_t T, int64_t N, int64_t P,
                    float* out, float* out_packed, cudaStream_t stream);
// order != null: the sorted copy (and out_search [T,N,3], AoS) holds the points in the order `order` [N] (search position ->
// caller point); `out` stays in caller order
// per-frame STR row order of the skinned cloud [T,N,3] and the search's copies in it (order.cu; N <= posed_order_max_points())
int posed_order_max_points();
int launch_posed_order(const float* skinned, int64_t T, int64_t N, int64_t n_pad, int32_t* row_order, int32_t* row_inv,
                       float* out_search, float* out_packed, unsigned char* perm, float* xq, cudaStream_t stream);
int launch_skin_fwd_sorted(const float* cano, const float* W, const float* R, const float* tr, int64_t T, int64_t N,
                           int64_t P, float* out, float* out_packed, unsigned char* perm, float* xq, int64_t n_pad,
                           cudaStream_t stream, const int32_t* order = nullptr, float* out_search = nullptr);
int64_t skin_bwd_workspace_floats(int64_t T, int64_t N, int64_t P);
int launch_skin_bwd(const float* cano, const float* W, const float* R, const float* tr, const float* g, int64_t T,
                    int64_t N, int64_t P, float* gW, float* gR, float* gtr, float* partials, cudaStream_t stream);

int launch_rot6d_fwd(const float* d6, int64_t B, float* R, cudaStream_t stream);
int launch_rot6d_bwd(const float* d6, const float* gR, int64_t B, float* gd6, cudaStream_t stream);
int launch_screw_fwd(const float* l, const float* m, const float* theta, const float* d, int64_t B, float* M,
                     cudaStream_t stream);
int launch_screw_bwd(const float* l, const float* m, const float* theta, const float* d, const float* gM, int64_t B,
                     float* gl, float* gm, float* gtheta, float* gd, cudaStream_t stream);

// Flattened joint tree for forward kinematics (utils/kinematic_utils.py:151-198).
struct FkParams {
    const float* axis;            // [E,3]
    const float* moment;          // [E,3]
    const float* theta;           // [T,E]
    const float* distance;        // [T,E] or null (=> d = 1e-6)
    const int32_t* order;         // [P] parts root-first (reverse_topo)
    const int32_t* parent;        // [P] parent part id, -1 for the root
    const int32_t* edge;          // [P] edge index joining part to its parent
    const int32_t* joint_type;    // [E] 0 as given, 1 revolute, 2 prismatic; or null
    int T, P;
};
int launch_fk_fwd(const FkParams& p, float* out, cudaStream_t stream);
int launch_fk_bwd(const FkParams& p, const float* fk, const float* g_out, float* gwork, float* g_axis, float* g_moment,
                  float* g_theta, float* g_dist, cudaStream_t stream);

// Fused loss + gradient of the bidirectional Chamfer energy from the search keys (energy.cu).
struct EnergyParams {
    const float* src;             // [B,N,3] skinned cloud
    const float* tgt;             // [B,M,3] observed frames
    const float* src_packed;      // packed copies (re-scan)
    const float* tgt_packed;
    const unsigned char* src_perm;      // [B,n_pad]: src_packed is x-sorted per 256-point block, perm = original offset
    const float* src_xq;                // [B,n_pad/256,16] quantile index of the sorted blocks
    const unsigned long long* keys_a;   // [B,N] row keys
    const unsigned long long* keys_b;   // [B,M] column keys
    int B, N, M, n_pad, m_pad;
    int row_chunk_pts, col_chunk_pts;
    float gscale;                 // upstream gradient of every per-point distance (1 for torch.sum)
    float* g_src;                 // [B,N,3], overwritten by the row pass
    double* loss;                 // [1]: sum of all per-point distances (written, not accumulated)
    long long* acc;               // [B,N,3] fixed-point accumulators of the reverse-direction terms, ZERO on entry
    const unsigned* col_bound;    // [1] float bits >= every column minimum (SymParams::col_bound)
    double* partials;             // [2 * energy_max_blocks()] per-block loss partials (no initialisation needed)
    unsigned* ticket;             // [1] ZERO on entry
    int32_t* nn_rows; int32_t* nn_cols;   // optional [B,N] / [B,M]: the arg-mins by caller index, the next evaluation's seeds
    float* d_fwd; int64_t* i_fwd; // optional [B,N]
    float* d_bwd; int64_t* i_bwd; // optional [B,M]
    // search in a permuted order (all null: the keys are in caller order).  The search ran on row_order / tgt_order copies
    // (src_packed, tgt_packed, keys and tie words are in that order); both passes still iterate in caller order.
    const int32_t* row_order;     // [N] or [B,N] (row_stride 0 / N): search position -> caller row
    const int32_t* row_inv;       // same shape: caller row -> search position
    int64_t row_stride;
    const int32_t* tgt_order;     // [B,M] per frame: search position -> caller target
    const int32_t* tgt_inv;       // [B,M]
    const unsigned* tie_a;        // [B,N] / [B,M] tie words of the search (SymParams::tie_a)
    const unsigned* tie_b;
    unsigned long long* ties;     // null, or [1]: += number of points resolved by the exact tie path
};
int energy_max_blocks();
int launch_energy_bwd(const EnergyParams& p, cudaStream_t stream);

int launch_knn(const float* ref, const float* query, int64_t B, int64_t n, int64_t m, int k, float* dist, int64_t* idx,
               int squared, cudaStream_t stream);
// windowed exact flow blend over x-sorted reference sets (knnk.cu)
int64_t flow_refs_sorted_floats(int64_t total_refs, int64_t T);
int launch_flow_refs_sort(const float* ref_cat, const int64_t* ref_off, int64_t T, int64_t max_refs, float* sorted,
                          int64_t* sorted_off, cudaStream_t stream);
int launch_knn3_blend_sorted(const float* query, const float* sorted, const int64_t* sorted_off, const float* flow_cat,
                             const int64_t* ref_off, int64_t T, int64_t m, int* qperm, float* blended,
                             unsigned char* mask, cudaStream_t stream);
int launch_knn3_blend(const float* query, const float* ref_cat, const float* flow_cat, const int64_t* ref_off,
                      int64_t T, int64_t m, float* blended, unsigned char* mask, cudaStream_t stream);

int launch_fps(const float* xyz, int64_t B, int64_t N, int64_t m, int* out, cudaStream_t stream);
int launch_fps_large(const float* xyz, int64_t B, int64_t N, int64_t m, float* temp, int* out, cudaStream_t stream);
int launch_ball_query(const float* new_xyz, const float* xyz, int64_t B, int64_t N, int64_t m, float radius,
                      int nsample, int* idx, cudaStream_t stream);

int launch_segmlp(const float* x, const float* w0, const float* b0, const float* w2, const float* glogits, int64_t N,
                  int64_t H, int64_t P, float* logits, float* gw0, float* gb0, float* gw2, cudaStream_t stream);
int launch_gumbel_st(const float* logits, const float* expo, const float* tau, const float* gW, int64_t N, int64_t P,
                     float* W, float* ysoft, float* glogits, cudaStream_t stream);

// Assignment loss (lap.cu): exact linear sum assignment per frame on on-the-fly Euclidean costs + matched-pair loss/grad.
int launch_lap(const float* src_base, const int64_t* src_idx, int64_t src_stride, const float* tgt, int64_t B, int64_t n,
               int* col4row, double* total, double* dual_u, int warm, cudaStream_t stream);
int launch_assign_loss_grad(const float* skinned, const int64_t* src_idx, const float* tgt, const int* col4row, int64_t T,
                            int64_t N, int64_t n, float lambda, float* g_skinned, int accumulate, double* loss,
                            cudaStream_t stream);

// Fused frame-independent head / tail of one relaxation iteration (relax.cu).
int launch_relax_head(const float* cano, const float* w0, const float* b0, const float* w2, const float* expo,
                      const int64_t* noise_index, const float* tau, const float* d6, int64_t N, int64_t H, int64_t P, int64_t T, float* logits,
                      float* W, float* ysoft, float* R, float* hot, cudaStream_t stream);
struct RelaxTail {
    const float* cano;            // [N,3]
    float* w0; float* b0; float* w2;              // seg MLP parameters [H,3], [H], [P,H] -- updated in place
    const float* ysoft;           // [N,P] soft assignment saved by the head
    const float* tau;             // [1]
    const float* gW;              // [N,P]  d loss / d W
    float* d6; float* tr;         // [T,P,6], [T,P,3] pose parameters -- updated in place
    const float* gR; const float* gtr;            // [T,P,9], [T,P,3]
    float* m_seg; float* v_seg;   // [4H + PH] Adam moments of [w0 | b0 | w2]
    float* m_d6; float* v_d6; float* m_tr; float* v_tr;
    float* step;                  // [1] completed optimisation steps (advanced by the kernel)
    float lr_pose, lr_seg, beta1, beta2, eps, wd;
    float* partials;              // [ceil(N/128)][4H + PH] per-chunk seg-gradient partials
    unsigned* tickets;            // [relax_tail_ticket_words(N)] zero before the FIRST call; the kernel re-arms them itself
    const double* loss_local;     // [1] this rank's loss
    float* bucket;                // [4H + PH + 1] reduced seg gradients + loss
    float* loss_out;              // [1] all-rank loss of the step
    const unsigned long long* peer_base; unsigned* epoch; int rank, world, n_pad;   // one-shot all-reduce (world > 1)
    int phase;                    // 0 everything; 1 gradients -> bucket only; 2 Adam from an (externally reduced) bucket
    int N, H, P, T;
};
int64_t relax_tail_workspace_floats(int64_t N, int64_t H, int64_t P);
int64_t relax_tail_ticket_words(int64_t N);
int launch_relax_tail(const RelaxTail& a, cudaStream_t stream);

// Fused head / tail of one kinematic-model iteration around the energy (kin.cu).
int launch_kin_head(const FkParams& p, const float* root_6d, const float* root_t, float* R, float* tr, float* fk,
                    cudaStream_t stream);
struct KinTail {
    const float* fk;              // [T,P,12] per-part poses before the root pose (kin_head)
    const float* gR; const float* gtr;            // [T,P,9], [T,P,3] d loss / d (R, tr) from the energy
    const double* loss_local;     // [1] this rank's loss
    const int32_t* order; const int32_t* parent; const int32_t* edge; const int32_t* joint_type;   // FkParams' tree
    float* axis; float* moment;   // [E,3] shared parameters -- updated in place
    float* theta; float* distance;                // [T,E]; distance may be null
    float* root_6d; float* root_t;                // [T,6], [T,3]; both null without a learned root pose
    float* grad;                  // [6E | loss | T*E theta | (T*E distance) | (6T root_6d, 3T root_t)]; [0, 6E] is the bucket
    float* m; float* v;           // Adam moments, same layout as grad (the loss slot is unused)
    float* step;                  // [1] completed optimisation steps (advanced by the kernel)
    float lr, beta1, beta2, eps, wd;
    float* partials;              // [kin_tail_workspace_floats(T,P)]
    float* loss_out;              // [1] all-rank loss of the step
    const unsigned long long* peer_base; unsigned* epoch; int rank, world, n_pad;   // one-shot all-reduce (world > 1)
    int phase;                    // 0 everything; 1 gradients only; 2 Adam from an (externally reduced) bucket
    int T, P;
};
int64_t kin_tail_workspace_floats(int64_t T, int64_t P);
int launch_kin_tail(const KinTail& a, cudaStream_t stream);
// Assignment loss of the kinematic model straight into the pose gradients (one-hot skinning weights).
struct KinAssign {
    const float* skinned;         // [T,N,3]
    const float* cano;            // [N,3]
    const int64_t* src_idx;       // [n] sampled canonical points
    const float* tgt;             // [T,n,3] sampled target points
    const int32_t* col4row;       // [T,n] target sample matched to source sample i
    const int32_t* sample_order;  // [n] sample indices grouped by part (stable)
    const int32_t* part_offsets;  // [P+1] part p owns sample_order[part_offsets[p] .. part_offsets[p+1])
    float lambda;
    float* gR; float* gtr;        // [T,P,9], [T,P,3]
    double* loss;                 // [1]
    int accumulate;               // add to gR / gtr / loss, else overwrite them
    double* partials;             // [kin_assign_blocks(T,P)]
    unsigned* ticket;             // [1] zero before the FIRST call; the kernel re-arms it
    int T, N, n, P;
};
int64_t kin_assign_blocks(int64_t T, int64_t P);
int launch_kin_assign(const KinAssign& a, cudaStream_t stream);
// Flow loss of the kinematic model straight into the pose gradients, on a window of the complete sequence.
struct KinFlow {
    const float* win;             // [K,N,3] consecutive complete frames
    const float* tflow;           // [K-1,N,3] blended target flow of pair k = (slot k, slot k+1)
    const uint8_t* mask;          // [K-1,N]
    const int32_t* slot_frame;    // [K] local frame of each slot, -1: canonical cloud or a neighbour rank's frame
    const float* cano;            // [N,3]
    const int32_t* point_order;   // [N] point indices grouped by part (stable)
    const int32_t* part_offsets;  // [P+1]
    float lambda;
    int robust;
    float* gR; float* gtr;        // [T,P,9], [T,P,3]
    double* loss;                 // [1]
    int accumulate;               // add to gR / gtr / loss, else overwrite them
    double* partials;             // [kin_flow_blocks(K,P)]
    unsigned* ticket;             // [1] zero before the FIRST call; the kernel re-arms it
    int K, N, P, T, q0, q1;       // the loss counts the pairs [q0, q1) of the window
};
int64_t kin_flow_blocks(int64_t K, int64_t P);
int launch_kin_flow(const KinFlow& a, cudaStream_t stream);
// Flow loss and its gradient w.r.t. the skinned cloud, per point, on a window of the complete sequence (flow.cu).
struct FlowGrad {
    const float* win;             // [K,N,3] consecutive complete frames
    const float* tflow;           // [K-1,N,3] blended target flow of pair k = (slot k, slot k+1)
    const uint8_t* mask;          // [K-1,N]
    const int32_t* slot_frame;    // [K] local frame of each slot, -1: canonical cloud or a neighbour rank's frame
    float lambda;
    int robust;
    float* g_skinned;             // [T,N,3]
    double* loss;                 // [1]
    int accumulate;               // add to g_skinned / loss, else overwrite them
    double* partials;             // [flow_grad_blocks(K,N)]
    unsigned* ticket;             // [1] zero before the FIRST call; the kernel re-arms it
    int K, N, T, q0, q1;          // the loss counts the pairs [q0, q1) of the window
};
int64_t flow_grad_blocks(int64_t K, int64_t N);
int launch_flow_grad(const FlowGrad& a, cudaStream_t stream);

int launch_allreduce_oneshot(const unsigned long long* peer_base, int rank, int world, int64_t n, int64_t n_pad,
                             unsigned* epoch, float* data, cudaStream_t stream);

int launch_probe(int variant, int iters, int blocks, const float* in, float* out, double* ms, double* ops_per_thread,
                 cudaStream_t stream);

}  // namespace reart
