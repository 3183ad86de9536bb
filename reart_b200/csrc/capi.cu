// capi.cu -- extern "C" boundary of libreart_b200.so (declared in include/reart_b200.h).
// Plain pointers and sizes only; argument validation and workspace carving live here, the
// kernels and their launchers in the other translation units (kernels.h).
#include "../../include/reart_b200.h"
#include "common.cuh"
#include "kernels.h"

using namespace reart;

namespace {

constexpr int64_t kAlign = 256;
inline int64_t align_up(int64_t v) { return round_up(v, kAlign); }
inline bool fits_int(int64_t v) { return v >= 0 && v <= 0x7fffffff; }

// The launch checks below read cudaGetLastError(): a NON-sticky error left behind by some other library on this thread
// (seen in practice after a CUPTI profiling session) must not be reported as ours, so every entry point starts by clearing it.
// A sticky error (a real fault) survives the clear and is still reported.
#define REART_ENTRY() (void)cudaGetLastError()

struct Carver {
    char* base;
    int64_t off;
    int64_t cap;
    bool ok;
    Carver(void* p, int64_t bytes) : base(static_cast<char*>(p)), off(0), cap(bytes), ok(p != nullptr || bytes == 0) {}
    template <typename T>
    T* take(int64_t count) {
        const int64_t bytes = align_up(count * (int64_t)sizeof(T));
        if (!ok || off + bytes > cap) { ok = false; return nullptr; }
        T* r = reinterpret_cast<T*>(base + off);
        off += bytes;
        return r;
    }
};

inline int64_t packed_bytes(int64_t B, int64_t P) { return align_up(B * packed_floats_per_batch(P) * 4); }
inline int64_t keys_bytes(int64_t B, int64_t P) { return align_up(B * P * 8); }
inline int64_t xq_floats(int64_t B, int64_t n_pad_sorted) { return B * (n_pad_sorted / kSortedChunk) * kQuantiles; }

}  // namespace

extern "C" {

const char* reart_version(void) { return "reart_b200 0.1.0 (sm_100a)"; }

const char* reart_last_cuda_error(void) {
    const int e = reart::last_cuda_error();
    return e ? cudaGetErrorString((cudaError_t)e) : "none";
}

const char* reart_error_string(int code) {
    switch (code) {
        case REART_OK: return "ok";
        case REART_ERR_INVALID_ARG: return "invalid argument (null pointer, negative or oversize dimension)";
        case REART_ERR_WORKSPACE: return "workspace too small or null";
        case REART_ERR_LAUNCH: return "CUDA launch or runtime error";
        case REART_ERR_UNSUPPORTED: return "unsupported size";
        default: return "unknown error";
    }
}

int64_t reart_knn1_workspace_bytes(int64_t B, int64_t P1, int64_t P2) {
    if (B < 0 || P1 < 0 || P2 < 0) return -1;
    return packed_bytes(B, P2) + keys_bytes(B, P1) + kAlign;
}

int reart_knn1_fwd(const float* p1, const float* p2, int64_t B, int64_t P1, int64_t P2, float* dists, int64_t* idx,
                   void* workspace, int64_t workspace_bytes, void* stream_) {
    REART_ENTRY();
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (B < 0 || P1 < 0 || P2 < 0 || !fits_int(B) || !fits_int(P1) || !fits_int(padded_points(P2)))
        return REART_ERR_INVALID_ARG;
    if (B == 0 || P1 == 0) return REART_OK;
    if (!p1 || !dists || !idx) return REART_ERR_INVALID_ARG;
    if (P2 == 0) {
        if (cudaMemsetAsync(dists, 0, sizeof(float) * (size_t)(B * P1), stream) != cudaSuccess) return REART_ERR_LAUNCH;
        if (cudaMemsetAsync(idx, 0, sizeof(int64_t) * (size_t)(B * P1), stream) != cudaSuccess) return REART_ERR_LAUNCH;
        return REART_OK;
    }
    if (!p2) return REART_ERR_INVALID_ARG;
    Carver ws(workspace, workspace_bytes);
    float* packed = ws.take<float>(B * packed_floats_per_batch(P2));
    u64* keys = ws.take<u64>(B * P1);
    if (!ws.ok) return REART_ERR_WORKSPACE;
    int rc = launch_pack_cloud(p2, packed, B, P2, stream);
    if (rc) return rc;
    KnnParams p = {};
    p.ndir = 1;
    p.B = (int)B;
    p.dir[0] = KnnDir{p1, packed, keys, dists, idx, (int)P1, (int)P2, (int)padded_points(P2), 0, 0, 0, kChunk, nullptr};
    rc = launch_knn1_search(p, stream);
    if (rc) return rc;
    return launch_knn1_finalize(p, stream);
}

int64_t reart_chamfer_workspace_bytes(int64_t B, int64_t N, int64_t M) {
    if (B < 0 || N < 0 || M < 0) return -1;
    return align_up(B * round_up(N, 256) * 12) + packed_bytes(B, M) + keys_bytes(B, N) + keys_bytes(B, M) +
           align_up(B * round_up(N, 256)) + align_up(xq_floats(B, round_up(N, 256)) * 4) + kAlign;
}

int reart_chamfer_bidir_fwd(const float* src, const float* tgt, int64_t B, int64_t N, int64_t M, float* d_fwd,
                            int64_t* i_fwd, float* d_bwd, int64_t* i_bwd, void* workspace, int64_t workspace_bytes,
                            void* stream_) {
    REART_ENTRY();
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (B < 0 || N < 0 || M < 0 || !fits_int(B) || !fits_int(padded_points(N)) || !fits_int(padded_points(M)))
        return REART_ERR_INVALID_ARG;
    if (B == 0) return REART_OK;
    if (N == 0 || M == 0) {
        // degenerate: each direction falls back to the zero-padding rule of the single search
        int rc = reart_knn1_fwd(src, tgt, B, N, M, d_fwd, i_fwd, workspace, workspace_bytes, stream_);
        if (rc) return rc;
        return reart_knn1_fwd(tgt, src, B, M, N, d_bwd, i_bwd, workspace, workspace_bytes, stream_);
    }
    if (!src || !tgt || !d_fwd || !i_fwd || !d_bwd || !i_bwd) return REART_ERR_INVALID_ARG;
    // src's packed copy is only read by the column-side index recovery: x-sorted per 256-point chunk
    const int64_t n_pad_sorted = round_up(N, 256);
    Carver ws(workspace, workspace_bytes);
    float* psrc = ws.take<float>(B * n_pad_sorted * 3);
    float* ptgt = ws.take<float>(B * packed_floats_per_batch(M));
    u64* kf = ws.take<u64>(B * N);
    u64* kb = ws.take<u64>(B * M);
    unsigned char* perm = ws.take<unsigned char>(B * n_pad_sorted);
    float* xq = ws.take<float>(xq_floats(B, n_pad_sorted));
    if (!ws.ok) return REART_ERR_WORKSPACE;
    int rc = launch_pack_cloud_sorted(src, psrc, perm, xq, B, N, n_pad_sorted, stream);
    if (rc) return rc;
    rc = launch_pack_cloud(tgt, ptgt, B, M, stream);
    if (rc) return rc;
    // One evaluation per (src_i, tgt_j) feeds both directions (chamfer_sym.cu).
    SymParams sp = {};
    sp.a = src; sp.b_packed = ptgt; sp.keys_a = kf; sp.keys_b = kb;
    sp.B = (int)B; sp.na = (int)N; sp.nb = (int)M; sp.nb_pad = (int)padded_points(M);
    sp.keys_one_allocation = 1;
    rc = launch_chamfer_sym(sp, stream);
    if (rc) return rc;
    if (sp.col_chunk_pts != 256) return REART_ERR_UNSUPPORTED;
    KnnParams p = {};
    p.ndir = 2;
    p.B = (int)B;
    p.dir[0] = KnnDir{src, ptgt, kf, d_fwd, i_fwd, (int)N, (int)M, (int)padded_points(M), 0, 0, 0, kChunk, nullptr};
    p.dir[1] = KnnDir{tgt, psrc, kb, d_bwd, i_bwd, (int)M, (int)N, (int)n_pad_sorted, 0, 0, 0, sp.col_chunk_pts, perm, xq};
    return launch_knn1_finalize(p, stream);
}

int reart_chamfer_sym_search(const float* src, const float* tgt_packed, int64_t B, int64_t N, int64_t M,
                             uint64_t* keys_a, uint64_t* keys_b, int32_t* col_chunk_pts, int variant, void* stream_) {
    REART_ENTRY();
    if (B <= 0 || N <= 0 || M <= 0 || !fits_int(B) || !fits_int(padded_points(N)) || !fits_int(padded_points(M)))
        return REART_ERR_INVALID_ARG;
    if (!src || !tgt_packed || !keys_a || !keys_b) return REART_ERR_INVALID_ARG;
    SymParams sp = {};
    sp.a = src; sp.b_packed = tgt_packed;
    sp.keys_a = reinterpret_cast<u64*>(keys_a); sp.keys_b = reinterpret_cast<u64*>(keys_b);
    sp.B = (int)B; sp.na = (int)N; sp.nb = (int)M; sp.nb_pad = (int)padded_points(M);
    sp.variant = variant;
    int rc = launch_chamfer_sym(sp, static_cast<cudaStream_t>(stream_));
    if (col_chunk_pts) *col_chunk_pts = sp.col_chunk_pts;
    return rc;
}

int reart_knn1_bwd(const float* p1, const float* p2, const int64_t* idx, const float* grad_dists, int64_t B,
                   int64_t P1, int64_t P2, float* grad_p1, float* grad_p2, void* stream_) {
    REART_ENTRY();
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (B < 0 || P1 < 0 || P2 < 0) return REART_ERR_INVALID_ARG;
    if (B == 0) return REART_OK;
    if ((P1 > 0 && (!p1 || !idx || !grad_dists || !grad_p1)) || (P2 > 0 && (!p2 || !grad_p2))) return REART_ERR_INVALID_ARG;
    return launch_knn1_bwd(p1, p2, idx, grad_dists, B, P1, P2, grad_p1, grad_p2, 0, stream);
}

int reart_chamfer_bidir_bwd(const float* src, const float* tgt, const int64_t* i_fwd, const int64_t* i_bwd,
                            const float* g_fwd, const float* g_bwd, int64_t B, int64_t N, int64_t M, float* grad_src,
                            float* grad_tgt, void* stream_) {
    REART_ENTRY();
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (B < 0 || N < 0 || M < 0) return REART_ERR_INVALID_ARG;
    if (B == 0) return REART_OK;
    if (N > 0 && M > 0 && (!src || !tgt || !i_fwd || !i_bwd || !g_fwd || !g_bwd || !grad_src)) return REART_ERR_INVALID_ARG;
    return launch_chamfer_bidir_bwd(src, tgt, i_fwd, i_bwd, g_fwd, g_bwd, B, N, M, grad_src, grad_tgt, stream);
}

int64_t reart_packed_bytes(int64_t B, int64_t P) {
    if (B < 0 || P < 0) return -1;
    return packed_bytes(B, P);
}

int reart_pack_cloud(const float* pts, int64_t B, int64_t P, float* packed, void* stream_) {
    REART_ENTRY();
    if (B < 0 || P < 0 || !fits_int(padded_points(P))) return REART_ERR_INVALID_ARG;
    if (B == 0) return REART_OK;
    if (!packed || (P > 0 && !pts)) return REART_ERR_INVALID_ARG;
    return launch_pack_cloud(pts, packed, B, P, static_cast<cudaStream_t>(stream_));
}

int reart_skin_fwd(const float* cano, const float* W, const float* R, const float* tr, int64_t T, int64_t N, int64_t P,
                   float* out, void* stream_) {
    REART_ENTRY();
    if (T < 0 || N < 0 || P < 0 || !fits_int(T) || !fits_int(N)) return REART_ERR_INVALID_ARG;
    if (T == 0 || N == 0) return REART_OK;
    if (!cano || !W || !R || !tr || !out) return REART_ERR_INVALID_ARG;
    return launch_skin_fwd(cano, W, R, tr, T, N, P, out, nullptr, static_cast<cudaStream_t>(stream_));
}

int64_t reart_skin_bwd_workspace_bytes(int64_t T, int64_t N, int64_t P) {
    if (T < 0 || N < 0 || P < 0) return -1;
    return align_up(skin_bwd_workspace_floats(T, N, P) * 4) + kAlign;
}

int reart_skin_bwd(const float* cano, const float* W, const float* R, const float* tr, const float* g, int64_t T,
                   int64_t N, int64_t P, float* gW, float* gR, float* gtr, void* workspace, int64_t workspace_bytes,
                   void* stream_) {
    REART_ENTRY();
    if (T < 0 || N < 0 || P < 0 || !fits_int(T) || !fits_int(N)) return REART_ERR_INVALID_ARG;
    if ((N * P > 0 && !gW) || (T * P > 0 && (!gR || !gtr))) return REART_ERR_INVALID_ARG;
    if (T > 0 && N > 0 && (!cano || !W || !R || !tr || !g)) return REART_ERR_INVALID_ARG;
    Carver ws(workspace, workspace_bytes);
    float* partials = ws.take<float>(skin_bwd_workspace_floats(T, N, P));
    if (!ws.ok) return REART_ERR_WORKSPACE;
    return launch_skin_bwd(cano, W, R, tr, g, T, N, P, gW, gR, gtr, partials, static_cast<cudaStream_t>(stream_));
}

int64_t reart_energy_workspace_bytes(int64_t T, int64_t N, int64_t M) {
    if (T < 0 || N < 0 || M < 0) return -1;
    return align_up(T * round_up(N, 256) * 12) + keys_bytes(T, N) + keys_bytes(T, M) + align_up(T * N * 12) +
           align_up(T * round_up(N, 256)) + align_up(xq_floats(T, round_up(N, 256)) * 4) +
           align_up(T * N * 24 + 64) + align_up(2 * (int64_t)energy_max_blocks() * 8) +
           align_up(skin_bwd_workspace_floats(T, N, 32) * 4) + align_up(T * (padded_points(M) / kChunk) * 32) +
           align_up(T * ceil_div(N, 256) * 4) + align_up(T * N * 12) + align_up(T * (N + M) * 4) + kAlign;
}

int reart_skinned_chamfer_fwd_bwd(const float* cano, const float* W, const float* R, const float* tr, const float* tgt,
                                  const float* tgt_packed, int64_t T, int64_t N, int64_t M, int64_t P, float* skinned,
                                  double* loss, float* gW, float* gR, float* gtr, float* g_skinned, int compute_grad,
                                  void* workspace, int64_t workspace_bytes, void* stream_) {
    REART_ENTRY();
    return reart_skinned_chamfer_fwd_bwd_ex(cano, W, R, tr, tgt, tgt_packed, T, N, M, P, skinned, loss, gW, gR, gtr, g_skinned,
                                            compute_grad, nullptr, nullptr, nullptr, nullptr, workspace, workspace_bytes, stream_);
}

int reart_skinned_chamfer_fwd_bwd_ex(const float* cano, const float* W, const float* R, const float* tr, const float* tgt,
                                     const float* tgt_packed, int64_t T, int64_t N, int64_t M, int64_t P, float* skinned,
                                     double* loss, float* gW, float* gR, float* gtr, float* g_skinned, int compute_grad,
                                     float* d_fwd, int64_t* i_fwd, float* d_bwd, int64_t* i_bwd, void* workspace,
                                     int64_t workspace_bytes, void* stream_) {
    REART_ENTRY();
    return reart_skinned_chamfer_fwd_bwd_culled(cano, W, R, tr, tgt, tgt_packed, T, N, M, P, skinned, loss, gW, gR, gtr, g_skinned,
                                                compute_grad, d_fwd, i_fwd, d_bwd, i_bwd, nullptr, nullptr, nullptr, workspace,
                                                workspace_bytes, stream_);
}

// The search order of reart_skinned_chamfer_fwd_bwd_ordered (null everywhere else).
struct SearchOrder {
    const int32_t* row_order; const int32_t* row_inv; const int32_t* tgt_order; const int32_t* tgt_inv;
    const float* tgt_search;      // [T,M,3] the observed frames in tgt_order (tgt_packed is then its packed copy)
};

static int energy_pipeline(const float* cano, const float* W, const float* hot, const float* R, const float* tr,
                           const float* tgt, const float* tgt_packed, int64_t T, int64_t N, int64_t M, int64_t P,
                           float* skinned, double* loss, float* gW, float* gR, float* gtr, float* g_skinned, int compute_grad,
                           float* d_fwd, int64_t* i_fwd, float* d_bwd, int64_t* i_bwd, int32_t* nn_rows, int32_t* nn_cols,
                           uint64_t* cull_stats, void* workspace, int64_t workspace_bytes, void* stream_,
                           const SearchOrder* order = nullptr);

int reart_skinned_chamfer_fwd_bwd_culled(const float* cano, const float* W, const float* R, const float* tr,
                                         const float* tgt, const float* tgt_packed, int64_t T, int64_t N, int64_t M,
                                         int64_t P, float* skinned, double* loss, float* gW, float* gR, float* gtr,
                                         float* g_skinned, int compute_grad, float* d_fwd, int64_t* i_fwd, float* d_bwd,
                                         int64_t* i_bwd, int32_t* nn_rows, int32_t* nn_cols, uint64_t* cull_stats,
                                         void* workspace, int64_t workspace_bytes, void* stream_) {
    REART_ENTRY();
    return energy_pipeline(cano, W, nullptr, R, tr, tgt, tgt_packed, T, N, M, P, skinned, loss, gW, gR, gtr, g_skinned,
                           compute_grad, d_fwd, i_fwd, d_bwd, i_bwd, nn_rows, nn_cols, cull_stats, workspace, workspace_bytes,
                           stream_);
}

int reart_skinned_chamfer_fwd_bwd_ordered(const float* cano, const float* W, const float* R, const float* tr,
                                          const float* tgt, const float* tgt_search, const float* tgt_search_packed,
                                          int64_t T, int64_t N, int64_t M, int64_t P, const int32_t* row_order,
                                          const int32_t* row_inv, const int32_t* tgt_order, const int32_t* tgt_inv,
                                          float* skinned, double* loss, float* gW, float* gR, float* gtr, float* g_skinned,
                                          int compute_grad, float* d_fwd, int64_t* i_fwd, float* d_bwd, int64_t* i_bwd,
                                          int32_t* nn_rows, int32_t* nn_cols, uint64_t* stats, void* workspace,
                                          int64_t workspace_bytes, void* stream_) {
    REART_ENTRY();
    if (!tgt_search || !row_order || !row_inv || !tgt_order || !tgt_inv || !nn_rows || !nn_cols) return REART_ERR_INVALID_ARG;
    const SearchOrder order = {row_order, row_inv, tgt_order, tgt_inv, tgt_search};
    return energy_pipeline(cano, W, nullptr, R, tr, tgt, tgt_search_packed, T, N, M, P, skinned, loss, gW, gR, gtr, g_skinned,
                           compute_grad, d_fwd, i_fwd, d_bwd, i_bwd, nn_rows, nn_cols, stats, workspace, workspace_bytes,
                           stream_, &order);
}

int reart_skinned_chamfer_fwd_bwd_fused(const float* cano, const float* hot, const float* W, const float* R,
                                        const float* tr, const float* tgt, const float* tgt_packed, int64_t T, int64_t N,
                                        int64_t M, int64_t P, float* skinned, double* loss, float* gW, float* gR,
                                        float* gtr, float* g_skinned, int compute_grad, void* workspace,
                                        int64_t workspace_bytes, void* stream_) {
    REART_ENTRY();
    if (!hot || (reinterpret_cast<uintptr_t>(hot) & 15) || (reinterpret_cast<uintptr_t>(cano) & 15) ||
        (reinterpret_cast<uintptr_t>(skinned) & 15))
        return REART_ERR_INVALID_ARG;
    return energy_pipeline(cano, W, hot, R, tr, tgt, tgt_packed, T, N, M, P, skinned, loss, gW, gR, gtr, g_skinned, compute_grad,
                           nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, workspace, workspace_bytes, stream_);
}

static int energy_pipeline(const float* cano, const float* W, const float* hot, const float* R, const float* tr,
                           const float* tgt, const float* tgt_packed, int64_t T, int64_t N, int64_t M, int64_t P,
                           float* skinned, double* loss, float* gW, float* gR, float* gtr, float* g_skinned, int compute_grad,
                           float* d_fwd, int64_t* i_fwd, float* d_bwd, int64_t* i_bwd, int32_t* nn_rows, int32_t* nn_cols,
                           uint64_t* cull_stats, void* workspace, int64_t workspace_bytes, void* stream_,
                           const SearchOrder* order) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (T <= 0 || N <= 0 || M <= 0 || P <= 0 || P > 32 || !fits_int(T) || !fits_int(padded_points(N)) ||
        !fits_int(padded_points(M)))
        return REART_ERR_INVALID_ARG;
    if (!cano || !W || !R || !tr || !tgt || !tgt_packed || !skinned || !loss) return REART_ERR_INVALID_ARG;
    if (compute_grad && (!gW || !gR || !gtr)) return REART_ERR_INVALID_ARG;
    // the skinned cloud's packed copy is x-sorted inside every 256-point column chunk (cheap index recovery)
    const int64_t n_pad_sorted = round_up(N, 256);
    Carver ws(workspace, workspace_bytes);
    float* psrc = ws.take<float>(T * n_pad_sorted * 3);
    u64* ka = ws.take<u64>(T * N);
    u64* kb = ws.take<u64>(T * M);
    float* gs = g_skinned ? g_skinned : ws.take<float>(T * N * 3);
    unsigned char* perm = ws.take<unsigned char>(T * n_pad_sorted);
    float* xq = ws.take<float>(xq_floats(T, n_pad_sorted));
    // [acc | ticket | col_bound]: the words that must be zero before the search, cleared by ONE memset
    const int64_t zero_bytes = T * N * 24 + 64;
    char* zero = ws.take<char>(zero_bytes);
    double* partials = ws.take<double>(2 * (int64_t)energy_max_blocks());
    float* bwd_partials = compute_grad ? ws.take<float>(skin_bwd_workspace_floats(T, N, P)) : nullptr;
    const bool cull = nn_rows != nullptr && nn_cols != nullptr;
    float* colbox = cull ? ws.take<float>(T * (padded_points(M) / kChunk) * 8) : nullptr;
    float* rowbound = cull ? ws.take<float>(T * ceil_div(N, 256)) : nullptr;
    // ordered search: the skinned rows in the search order, and the tie words [T,N] | [T,M] of both sides
    float* skinned_search = order ? ws.take<float>(T * N * 3) : nullptr;
    unsigned* tie = order ? ws.take<unsigned>(T * (N + M)) : nullptr;
    if (!ws.ok) return REART_ERR_WORKSPACE;
    long long* acc = reinterpret_cast<long long*>(zero);
    unsigned* ticket = reinterpret_cast<unsigned*>(zero + T * N * 24);
    unsigned* col_bound = ticket + 1;
    if (cudaMemsetAsync(zero, 0, (size_t)zero_bytes, stream) != cudaSuccess) return REART_ERR_LAUNCH;
    int rc = kOk;
    SymParams sp = {};
    sp.a = skinned; sp.b_packed = tgt_packed; sp.keys_a = ka; sp.keys_b = kb;
    sp.B = (int)T; sp.na = (int)N; sp.nb = (int)M; sp.nb_pad = (int)padded_points(M);
    sp.col_bound = col_bound;
    sp.keys_one_allocation = 1;
    if (hot) {
        // fused producer: the search skins its own rows and emits the cloud + x-sorted copy as by-products (no skin launch)
        if (cull) return REART_ERR_INVALID_ARG;
        sp.sk_cano = cano; sp.sk_hot = hot; sp.sk_R = R; sp.sk_tr = tr; sp.sk_P = (int)P; sp.sk_npad = (int)n_pad_sorted;
        sp.sk_out = skinned; sp.sk_sorted = psrc; sp.sk_perm = perm; sp.sk_xq = xq;
    } else {
        rc = launch_skin_fwd_sorted(cano, W, R, tr, T, N, P, skinned, psrc, perm, xq, n_pad_sorted, stream,
                                    order ? order->row_order : nullptr, skinned_search);
        if (rc) return rc;
    }
    if (order) {
        sp.a = skinned_search;
        sp.tie_a = tie; sp.tie_b = tie + T * N;
    }
    if (cull) {
        // seeds = the arg-mins of the previous evaluation (nn_* = -1: none, brute force); bounds, then the culled search
        CullParams cp = {};
        cp.a = sp.a; cp.b = order ? order->tgt_search : tgt; cp.nn_rows = nn_rows; cp.nn_cols = nn_cols;
        cp.B = (int)T; cp.na = (int)N; cp.nb = (int)M; cp.nb_pad = (int)padded_points(M);
        cp.colbox = colbox; cp.rowbound = rowbound;
        cp.coarse = (N >= 8192 && M >= 8192 && N <= 800000 && M <= 800000) ? 1 : 0;   // small clouds: the pass costs more than it saves
        rc = launch_cull_bounds(cp, stream);
        if (rc) return rc;
        sp.cull = 1; sp.colbox = colbox; sp.rowbound = rowbound;
        sp.cull_stats = reinterpret_cast<unsigned long long*>(cull_stats);
    }
    rc = launch_chamfer_sym(sp, stream);
    if (rc) return rc;
    EnergyParams ep = {};
    ep.src = skinned; ep.tgt = tgt; ep.src_packed = psrc; ep.tgt_packed = tgt_packed; ep.keys_a = ka; ep.keys_b = kb;
    ep.B = (int)T; ep.N = (int)N; ep.M = (int)M; ep.n_pad = (int)n_pad_sorted; ep.m_pad = (int)padded_points(M);
    ep.row_chunk_pts = kChunk; ep.col_chunk_pts = sp.col_chunk_pts; ep.gscale = 1.0f; ep.g_src = gs; ep.loss = loss;
    if (sp.col_chunk_pts != 256) return REART_ERR_UNSUPPORTED;       // the sorted copy is built per 256-point chunk
    ep.d_fwd = d_fwd; ep.i_fwd = i_fwd; ep.d_bwd = d_bwd; ep.i_bwd = i_bwd;
    ep.nn_rows = nn_rows; ep.nn_cols = nn_cols;                      // the next evaluation's seeds
    ep.src_perm = perm; ep.src_xq = xq; ep.acc = acc; ep.col_bound = col_bound; ep.partials = partials; ep.ticket = ticket;
    if (order) {
        ep.row_order = order->row_order; ep.row_inv = order->row_inv; ep.tgt_order = order->tgt_order; ep.tgt_inv = order->tgt_inv;
        ep.tie_a = sp.tie_a; ep.tie_b = sp.tie_b;
        ep.ties = cull_stats ? reinterpret_cast<unsigned long long*>(cull_stats) + 2 : nullptr;
    }
    rc = launch_energy_bwd(ep, stream);
    if (rc || !compute_grad) return rc;
    return launch_skin_bwd(cano, W, R, tr, gs, T, N, P, gW, gR, gtr, bwd_partials, stream);
}

int reart_segmlp_fwd(const float* x, const float* w0, const float* b0, const float* w2, int64_t N, int64_t H, int64_t P,
                     float* logits, void* stream_) {
    REART_ENTRY();
    if (N < 0 || H <= 0 || P <= 0) return REART_ERR_INVALID_ARG;
    if (N == 0) return REART_OK;
    if (!x || !w0 || !b0 || !w2 || !logits) return REART_ERR_INVALID_ARG;
    return launch_segmlp(x, w0, b0, w2, nullptr, N, H, P, logits, nullptr, nullptr, nullptr,
                         static_cast<cudaStream_t>(stream_));
}

int reart_segmlp_bwd(const float* x, const float* w0, const float* b0, const float* w2, const float* glogits, int64_t N,
                     int64_t H, int64_t P, float* gw0, float* gb0, float* gw2, void* stream_) {
    REART_ENTRY();
    if (N < 0 || H <= 0 || P <= 0 || !gw0 || !gb0 || !gw2) return REART_ERR_INVALID_ARG;
    if (N > 0 && (!x || !w0 || !b0 || !w2 || !glogits)) return REART_ERR_INVALID_ARG;
    if (N == 0) {
        cudaStream_t st = static_cast<cudaStream_t>(stream_);
        if (cudaMemsetAsync(gw0, 0, sizeof(float) * (size_t)H * 3, st) != cudaSuccess) return REART_ERR_LAUNCH;
        if (cudaMemsetAsync(gb0, 0, sizeof(float) * (size_t)H, st) != cudaSuccess) return REART_ERR_LAUNCH;
        if (cudaMemsetAsync(gw2, 0, sizeof(float) * (size_t)H * P, st) != cudaSuccess) return REART_ERR_LAUNCH;
        return REART_OK;
    }
    return launch_segmlp(x, w0, b0, w2, glogits, N, H, P, nullptr, gw0, gb0, gw2, static_cast<cudaStream_t>(stream_));
}

int reart_gumbel_st_fwd(const float* logits, const float* expo, const float* tau, int64_t N, int64_t P, float* W,
                        float* ysoft, void* stream_) {
    REART_ENTRY();
    if (N < 0 || P <= 0) return REART_ERR_INVALID_ARG;
    if (N == 0) return REART_OK;
    if (!logits || !expo || !tau || !W || !ysoft) return REART_ERR_INVALID_ARG;
    return launch_gumbel_st(logits, expo, tau, nullptr, N, P, W, ysoft, nullptr, static_cast<cudaStream_t>(stream_));
}

int reart_gumbel_st_bwd(const float* ysoft, const float* tau, const float* gW, int64_t N, int64_t P, float* glogits,
                        void* stream_) {
    REART_ENTRY();
    if (N < 0 || P <= 0) return REART_ERR_INVALID_ARG;
    if (N == 0) return REART_OK;
    if (!ysoft || !tau || !gW || !glogits) return REART_ERR_INVALID_ARG;
    return launch_gumbel_st(nullptr, nullptr, tau, gW, N, P, nullptr, const_cast<float*>(ysoft), glogits,
                            static_cast<cudaStream_t>(stream_));
}

int reart_relax_head(const float* cano, const float* w0, const float* b0, const float* w2, const float* expo,
                     const int64_t* noise_index, const float* tau, const float* d6, int64_t N, int64_t H, int64_t P, int64_t T, float* logits,
                     float* W, float* ysoft, float* R, float* hot, void* stream_) {
    REART_ENTRY();
    if (N < 0 || T < 0 || H <= 0 || P <= 0 || !fits_int(4 * N) || !fits_int(T * P)) return REART_ERR_INVALID_ARG;
    if (hot && (reinterpret_cast<uintptr_t>(hot) & 15)) return REART_ERR_INVALID_ARG;
    if (N > 0 && (!cano || !w0 || !b0 || !w2 || !expo || !tau || !W || !ysoft)) return REART_ERR_INVALID_ARG;
    if (T > 0 && (!d6 || !R)) return REART_ERR_INVALID_ARG;
    return launch_relax_head(cano, w0, b0, w2, expo, noise_index, tau, d6, N, H, P, T, logits, W, ysoft, R, hot,
                             static_cast<cudaStream_t>(stream_));
}

int64_t reart_relax_tail_workspace_bytes(int64_t N, int64_t H, int64_t P) {
    if (N < 0 || H <= 0 || P <= 0) return -1;
    return align_up(relax_tail_workspace_floats(N, H, P) * 4) + kAlign;
}

int64_t reart_relax_tail_ticket_words(int64_t N) { return N < 0 ? -1 : relax_tail_ticket_words(N); }

int reart_relax_tail(const reart_relax_tail_args* x, void* stream_) {
    REART_ENTRY();
    if (!x || x->N <= 0 || x->T <= 0 || x->H <= 0 || x->P <= 0 || !fits_int(x->N) || !fits_int(x->T * x->P))
        return REART_ERR_INVALID_ARG;
    if (!x->cano || !x->w0 || !x->b0 || !x->w2 || !x->ysoft || !x->tau || !x->gW || !x->d6 || !x->tr || !x->gR || !x->gtr ||
        !x->m_seg || !x->v_seg || !x->m_d6 || !x->v_d6 || !x->m_tr || !x->v_tr || !x->step || !x->partials || !x->tickets ||
        !x->loss_local || !x->bucket || !x->loss_out || x->phase < 0 || x->phase > 2 || x->world < 1 || x->rank < 0 ||
        x->rank >= x->world)
        return REART_ERR_INVALID_ARG;
    RelaxTail a = {};
    a.cano = x->cano; a.w0 = x->w0; a.b0 = x->b0; a.w2 = x->w2; a.ysoft = x->ysoft; a.tau = x->tau; a.gW = x->gW;
    a.d6 = x->d6; a.tr = x->tr; a.gR = x->gR; a.gtr = x->gtr;
    a.m_seg = x->m_seg; a.v_seg = x->v_seg; a.m_d6 = x->m_d6; a.v_d6 = x->v_d6; a.m_tr = x->m_tr; a.v_tr = x->v_tr;
    a.step = x->step; a.lr_pose = x->lr_pose; a.lr_seg = x->lr_seg; a.beta1 = x->beta1; a.beta2 = x->beta2; a.eps = x->eps;
    a.wd = x->weight_decay; a.partials = x->partials; a.tickets = x->tickets; a.loss_local = x->loss_local;
    a.bucket = x->bucket; a.loss_out = x->loss_out;
    a.peer_base = reinterpret_cast<const unsigned long long*>(x->peer_base); a.epoch = x->epoch;
    a.rank = x->rank; a.world = x->world; a.n_pad = x->n_pad; a.phase = x->phase;
    a.N = (int)x->N; a.H = (int)x->H; a.P = (int)x->P; a.T = (int)x->T;
    return launch_relax_tail(a, static_cast<cudaStream_t>(stream_));
}

int reart_kin_head(const float* axis, const float* moment, const float* theta, const float* distance, const int32_t* order,
                   const int32_t* parent, const int32_t* edge, const int32_t* joint_type, const float* root_6d,
                   const float* root_t, int64_t T, int64_t P, float* R, float* tr, float* fk, void* stream_) {
    REART_ENTRY();
    if (T < 0 || P < 1 || !fits_int(T * P * 12)) return REART_ERR_INVALID_ARG;
    if (P > 32) return REART_ERR_UNSUPPORTED;
    if (T == 0) return REART_OK;
    if (!order || !parent || !edge || !R || !tr || !fk || (P > 1 && (!axis || !moment || !theta)) || (!root_6d != !root_t))
        return REART_ERR_INVALID_ARG;
    FkParams p = {axis, moment, theta, distance, order, parent, edge, joint_type, (int)T, (int)P};
    return launch_kin_head(p, root_6d, root_t, R, tr, fk, static_cast<cudaStream_t>(stream_));
}

int64_t reart_kin_tail_workspace_bytes(int64_t T, int64_t P) {
    if (T < 0 || P < 1) return -1;
    return align_up(kin_tail_workspace_floats(T, P) * 4) + kAlign;
}

int reart_kin_tail(const reart_kin_tail_args* x, void* stream_) {
    REART_ENTRY();
    if (!x || x->T <= 0 || x->P < 1 || !fits_int(x->T * x->P * 12)) return REART_ERR_INVALID_ARG;
    if (x->P > 32) return REART_ERR_UNSUPPORTED;
    // a one-part model has no joints (E = 0): axis, moment and theta may be null there, as in reart_kin_head
    if (!x->fk || !x->gR || !x->gtr || !x->loss_local || !x->order || !x->parent || !x->edge ||
        (x->P > 1 && (!x->axis || !x->moment || !x->theta)) || (!x->root_6d != !x->root_t) || !x->grad || !x->m || !x->v || !x->step ||
        !x->partials || !x->loss_out || x->phase < 0 || x->phase > 2 || x->world < 1 || x->rank < 0 || x->rank >= x->world)
        return REART_ERR_INVALID_ARG;
    KinTail a = {};
    a.fk = x->fk; a.gR = x->gR; a.gtr = x->gtr; a.loss_local = x->loss_local;
    a.order = x->order; a.parent = x->parent; a.edge = x->edge; a.joint_type = x->joint_type;
    a.axis = x->axis; a.moment = x->moment; a.theta = x->theta; a.distance = x->distance;
    a.root_6d = x->root_6d; a.root_t = x->root_t;
    a.grad = x->grad; a.m = x->m; a.v = x->v; a.step = x->step;
    a.lr = x->lr; a.beta1 = x->beta1; a.beta2 = x->beta2; a.eps = x->eps; a.wd = x->weight_decay;
    a.partials = x->partials; a.loss_out = x->loss_out;
    a.peer_base = reinterpret_cast<const unsigned long long*>(x->peer_base); a.epoch = x->epoch;
    a.rank = x->rank; a.world = x->world; a.n_pad = x->n_pad; a.phase = x->phase;
    a.T = (int)x->T; a.P = (int)x->P;
    return launch_kin_tail(a, static_cast<cudaStream_t>(stream_));
}

int64_t reart_kin_assign_workspace_bytes(int64_t T, int64_t P) {
    if (T < 0 || P < 1 || P > 32) return -1;
    return align_up(kin_assign_blocks(T, P) * 8) + align_up(4) + kAlign;
}

int reart_kin_assign(const float* skinned, const float* cano, const int64_t* src_idx, const float* tgt,
                     const int32_t* col4row, const int32_t* sample_order, const int32_t* part_offsets, float lambda, int64_t T,
                     int64_t N, int64_t n, int64_t P, float* gR, float* gtr, double* loss, int accumulate, void* workspace,
                     int64_t workspace_bytes, void* stream_) {
    REART_ENTRY();
    if (T < 0 || N < 0 || n < 0 || P < 1 || !fits_int(T * P * 12) || !fits_int(T * N * 3) || !fits_int(T * n * 3))
        return REART_ERR_INVALID_ARG;
    if (P > 32) return REART_ERR_UNSUPPORTED;
    if (T == 0) return REART_OK;
    if (n == 0 || N == 0 || !skinned || !cano || !src_idx || !tgt || !col4row || !sample_order || !part_offsets || !gR ||
        !gtr || !loss)
        return REART_ERR_INVALID_ARG;
    Carver ws(workspace, workspace_bytes);
    double* partials = ws.take<double>(kin_assign_blocks(T, P));
    unsigned* ticket = ws.take<unsigned>(1);
    if (!ws.ok) return REART_ERR_WORKSPACE;
    KinAssign a = {};
    a.skinned = skinned; a.cano = cano; a.src_idx = src_idx; a.tgt = tgt; a.col4row = col4row;
    a.sample_order = sample_order; a.part_offsets = part_offsets; a.lambda = lambda;
    a.gR = gR; a.gtr = gtr; a.loss = loss; a.accumulate = accumulate ? 1 : 0;
    a.partials = partials; a.ticket = ticket;
    a.T = (int)T; a.N = (int)N; a.n = (int)n; a.P = (int)P;
    return launch_kin_assign(a, static_cast<cudaStream_t>(stream_));
}

int64_t reart_kin_flow_workspace_bytes(int64_t K, int64_t P) {
    if (K < 2 || P < 1 || P > 32) return -1;
    return align_up(kin_flow_blocks(K, P) * 8) + align_up(4) + kAlign;
}

int reart_kin_flow(const float* win, const float* tflow, const uint8_t* mask, const int32_t* slot_frame, const float* cano,
                   const int32_t* point_order, const int32_t* part_offsets, float lambda, int robust, int64_t K, int64_t N,
                   int64_t P, int64_t T, int64_t q0, int64_t q1, float* gR, float* gtr, double* loss, int accumulate,
                   void* workspace, int64_t workspace_bytes, void* stream_) {
    REART_ENTRY();
    if (T < 0 || K < 0 || N < 0 || P < 1 || !fits_int(T * P * 12) || !fits_int(K * N * 3) || !fits_int(K * P))
        return REART_ERR_INVALID_ARG;
    if (P > 32) return REART_ERR_UNSUPPORTED;
    if (T == 0) return REART_OK;
    if (K < 2 || N == 0 || q0 < 0 || q1 < q0 || q1 > K - 1) return REART_ERR_INVALID_ARG;
    if (!win || !tflow || !mask || !slot_frame || !cano || !point_order || !part_offsets || !gR || !gtr || !loss)
        return REART_ERR_INVALID_ARG;
    Carver ws(workspace, workspace_bytes);
    double* partials = ws.take<double>(kin_flow_blocks(K, P));
    unsigned* ticket = ws.take<unsigned>(1);
    if (!ws.ok) return REART_ERR_WORKSPACE;
    KinFlow a = {};
    a.win = win; a.tflow = tflow; a.mask = mask; a.slot_frame = slot_frame; a.cano = cano;
    a.point_order = point_order; a.part_offsets = part_offsets; a.lambda = lambda; a.robust = robust ? 1 : 0;
    a.gR = gR; a.gtr = gtr; a.loss = loss; a.accumulate = accumulate ? 1 : 0;
    a.partials = partials; a.ticket = ticket;
    a.K = (int)K; a.N = (int)N; a.P = (int)P; a.T = (int)T; a.q0 = (int)q0; a.q1 = (int)q1;
    return launch_kin_flow(a, static_cast<cudaStream_t>(stream_));
}

int64_t reart_flow_grad_workspace_bytes(int64_t K, int64_t N) {
    if (K < 2 || N < 1 || !fits_int(K * N * 3)) return -1;
    return align_up(flow_grad_blocks(K, N) * 8) + align_up(4) + kAlign;
}

int reart_flow_grad(const float* win, const float* tflow, const uint8_t* mask, const int32_t* slot_frame, float lambda,
                    int robust, int64_t K, int64_t N, int64_t T, int64_t q0, int64_t q1, float* g_skinned, double* loss,
                    int accumulate, void* workspace, int64_t workspace_bytes, void* stream_) {
    REART_ENTRY();
    if (T < 0 || K < 0 || N < 0 || !fits_int(K * N * 3) || !fits_int(T * N * 3)) return REART_ERR_INVALID_ARG;
    if (T == 0) return REART_OK;
    if (K < 2 || N == 0 || q0 < 0 || q1 < q0 || q1 > K - 1) return REART_ERR_INVALID_ARG;
    if (!win || !tflow || !mask || !slot_frame || !g_skinned || !loss) return REART_ERR_INVALID_ARG;
    Carver ws(workspace, workspace_bytes);
    double* partials = ws.take<double>(flow_grad_blocks(K, N));
    unsigned* ticket = ws.take<unsigned>(1);
    if (!ws.ok) return REART_ERR_WORKSPACE;
    FlowGrad a = {};
    a.win = win; a.tflow = tflow; a.mask = mask; a.slot_frame = slot_frame;
    a.lambda = lambda; a.robust = robust ? 1 : 0;
    a.g_skinned = g_skinned; a.loss = loss; a.accumulate = accumulate ? 1 : 0;
    a.partials = partials; a.ticket = ticket;
    a.K = (int)K; a.N = (int)N; a.T = (int)T; a.q0 = (int)q0; a.q1 = (int)q1;
    return launch_flow_grad(a, static_cast<cudaStream_t>(stream_));
}

int reart_rot6d_fwd(const float* d6, int64_t B, float* R, void* stream_) {
    REART_ENTRY();
    if (B < 0) return REART_ERR_INVALID_ARG;
    if (B == 0) return REART_OK;
    if (!d6 || !R) return REART_ERR_INVALID_ARG;
    return launch_rot6d_fwd(d6, B, R, static_cast<cudaStream_t>(stream_));
}

int reart_rot6d_bwd(const float* d6, const float* gR, int64_t B, float* gd6, void* stream_) {
    REART_ENTRY();
    if (B < 0) return REART_ERR_INVALID_ARG;
    if (B == 0) return REART_OK;
    if (!d6 || !gR || !gd6) return REART_ERR_INVALID_ARG;
    return launch_rot6d_bwd(d6, gR, B, gd6, static_cast<cudaStream_t>(stream_));
}

int reart_screw_to_transform_fwd(const float* l, const float* m, const float* theta, const float* d, int64_t B,
                                 float* M, void* stream_) {
    REART_ENTRY();
    if (B < 0) return REART_ERR_INVALID_ARG;
    if (B == 0) return REART_OK;
    if (!l || !m || !theta || !d || !M) return REART_ERR_INVALID_ARG;
    return launch_screw_fwd(l, m, theta, d, B, M, static_cast<cudaStream_t>(stream_));
}

int reart_screw_to_transform_bwd(const float* l, const float* m, const float* theta, const float* d, const float* gM,
                                 int64_t B, float* gl, float* gm, float* gtheta, float* gd, void* stream_) {
    REART_ENTRY();
    if (B < 0) return REART_ERR_INVALID_ARG;
    if (B == 0) return REART_OK;
    if (!l || !m || !theta || !d || !gM || !gl || !gm || !gtheta || !gd) return REART_ERR_INVALID_ARG;
    return launch_screw_bwd(l, m, theta, d, gM, B, gl, gm, gtheta, gd, static_cast<cudaStream_t>(stream_));
}

int reart_fk_fwd(const float* axis, const float* moment, const float* theta, const float* distance,
                 const int32_t* order, const int32_t* parent, const int32_t* edge, const int32_t* joint_type, int64_t T,
                 int64_t P, float* out, void* stream_) {
    REART_ENTRY();
    if (T < 0 || P < 0 || !fits_int(T) || !fits_int(P)) return REART_ERR_INVALID_ARG;
    if (T == 0 || P == 0) return REART_OK;
    if (!order || !parent || !edge || !out || (P > 1 && (!axis || !moment || !theta))) return REART_ERR_INVALID_ARG;
    FkParams p = {axis, moment, theta, distance, order, parent, edge, joint_type, (int)T, (int)P};
    return launch_fk_fwd(p, out, static_cast<cudaStream_t>(stream_));
}

int reart_fk_bwd(const float* axis, const float* moment, const float* theta, const float* distance,
                 const int32_t* order, const int32_t* parent, const int32_t* edge, const int32_t* joint_type, int64_t T,
                 int64_t P, const float* fk_out, const float* g_out, float* g_axis, float* g_moment, float* g_theta,
                 float* g_dist, float* workspace, void* stream_) {
    REART_ENTRY();
    if (T < 0 || P < 0 || !fits_int(T) || !fits_int(P)) return REART_ERR_INVALID_ARG;
    if (T == 0 || P <= 1) return REART_OK;
    if (!order || !parent || !edge || !fk_out || !g_out || !axis || !moment || !theta || !g_axis || !g_moment ||
        !g_theta || !workspace)
        return REART_ERR_INVALID_ARG;
    FkParams p = {axis, moment, theta, distance, order, parent, edge, joint_type, (int)T, (int)P};
    return launch_fk_bwd(p, fk_out, g_out, workspace, g_axis, g_moment, g_theta, distance ? g_dist : nullptr,
                         static_cast<cudaStream_t>(stream_));
}

int reart_knn(const float* ref, const float* query, int64_t B, int64_t n, int64_t m, int k, float* dist, int64_t* idx,
              void* stream_) {
    REART_ENTRY();
    if (B < 0 || n < 0 || m < 0 || k < 1 || k > 8 || !fits_int(n) || !fits_int(m)) return REART_ERR_INVALID_ARG;
    if (B == 0 || m == 0) return REART_OK;
    if (n < k) return REART_ERR_INVALID_ARG;
    if (!ref || !query || !dist || !idx) return REART_ERR_INVALID_ARG;
    return launch_knn(ref, query, B, n, m, k, dist, idx, 0, static_cast<cudaStream_t>(stream_));
}

int reart_knn_sq(const float* ref, const float* query, int64_t B, int64_t n, int64_t m, int k, float* dist, int64_t* idx,
                 void* stream_) {
    REART_ENTRY();
    if (B < 0 || n < 0 || m < 0 || k < 1 || k > 8 || !fits_int(n) || !fits_int(m)) return REART_ERR_INVALID_ARG;
    if (B == 0 || m == 0) return REART_OK;
    if (n < k) return REART_ERR_INVALID_ARG;
    if (!ref || !query || !dist || !idx) return REART_ERR_INVALID_ARG;
    return launch_knn(ref, query, B, n, m, k, dist, idx, 1, static_cast<cudaStream_t>(stream_));
}

int reart_knn3_blend(const float* query, const float* ref_cat, const float* flow_cat, const int64_t* ref_offsets,
                     int64_t T, int64_t m, float* blended, uint8_t* mask, void* stream_) {
    REART_ENTRY();
    if (T < 0 || m < 0 || !fits_int(m)) return REART_ERR_INVALID_ARG;
    if (T == 0 || m == 0) return REART_OK;
    if (!query || !ref_cat || !flow_cat || !ref_offsets || !blended) return REART_ERR_INVALID_ARG;
    return launch_knn3_blend(query, ref_cat, flow_cat, ref_offsets, T, m, blended, mask,
                             static_cast<cudaStream_t>(stream_));
}

int64_t reart_flow_refs_sorted_bytes(int64_t total_refs, int64_t T) {
    if (total_refs < 0 || T < 0) return 0;
    return flow_refs_sorted_floats(total_refs, T) * (int64_t)sizeof(float);
}

int reart_flow_refs_sort(const float* ref_cat, const int64_t* ref_offsets, int64_t T, int64_t max_refs, void* sorted,
                         int64_t sorted_bytes, int64_t total_refs, int64_t* sorted_offsets, void* stream_) {
    REART_ENTRY();
    if (T < 0 || max_refs < 0 || total_refs < 0) return REART_ERR_INVALID_ARG;
    if (T == 0) return REART_OK;
    if (!ref_cat || !ref_offsets || !sorted || !sorted_offsets) return REART_ERR_INVALID_ARG;
    if (sorted_bytes < reart_flow_refs_sorted_bytes(total_refs, T)) return REART_ERR_WORKSPACE;
    return launch_flow_refs_sort(ref_cat, ref_offsets, T, max_refs, static_cast<float*>(sorted), sorted_offsets,
                                 static_cast<cudaStream_t>(stream_));
}

int reart_knn3_blend_sorted(const float* query, const void* sorted, const int64_t* sorted_offsets, const float* flow_cat,
                            const int64_t* ref_offsets, int64_t T, int64_t m, int32_t* query_order, float* blended,
                            uint8_t* mask, void* stream_) {
    REART_ENTRY();
    if (T < 0 || m < 0 || !fits_int(m)) return REART_ERR_INVALID_ARG;
    if (T == 0 || m == 0) return REART_OK;
    if (!query || !sorted || !sorted_offsets || !flow_cat || !ref_offsets || !query_order || !blended) return REART_ERR_INVALID_ARG;
    return launch_knn3_blend_sorted(query, static_cast<const float*>(sorted), sorted_offsets, flow_cat, ref_offsets, T, m,
                                    query_order, blended, mask, static_cast<cudaStream_t>(stream_));
}

int reart_lap(const float* src, const int64_t* src_idx, int64_t src_points, const float* tgt, int64_t B, int64_t n,
              int32_t* col4row, double* total, double* dual_u, int warm_start, void* stream_) {
    REART_ENTRY();
    if (B < 0 || n < 0 || src_points < 0) return REART_ERR_INVALID_ARG;
    if (B == 0 || n == 0) return REART_OK;
    if (!src || !tgt || !col4row || (!src_idx && src_points < n)) return REART_ERR_INVALID_ARG;
    if (n > 4096) return REART_ERR_UNSUPPORTED;
    return launch_lap(src, src_idx, src_points * 3, tgt, B, n, col4row, total, dual_u, warm_start && dual_u ? 1 : 0,
                      static_cast<cudaStream_t>(stream_));
}

int reart_assign_loss_grad(const float* skinned, const int64_t* src_idx, const float* tgt, const int32_t* col4row, int64_t T,
                           int64_t N, int64_t n, float lambda, float* g_skinned, int accumulate, double* loss,
                           void* stream_) {
    REART_ENTRY();
    if (T < 0 || N < 0 || n < 0) return REART_ERR_INVALID_ARG;
    if (T == 0 || n == 0) return REART_OK;
    if (!skinned || !src_idx || !tgt || !col4row || !loss) return REART_ERR_INVALID_ARG;
    return launch_assign_loss_grad(skinned, src_idx, tgt, col4row, T, N, n, lambda, g_skinned, accumulate, loss,
                                   static_cast<cudaStream_t>(stream_));
}

int reart_fps(const float* xyz, int64_t B, int64_t N, int64_t npoint, int32_t* out, void* stream_) {
    REART_ENTRY();
    if (B < 0 || N < 0 || npoint < 0) return REART_ERR_INVALID_ARG;
    if (B == 0 || npoint == 0) return REART_OK;
    if (!xyz || !out || N == 0) return REART_ERR_INVALID_ARG;
    return launch_fps(xyz, B, N, npoint, out, static_cast<cudaStream_t>(stream_));
}

int reart_fps_temp(const float* xyz, int64_t B, int64_t N, int64_t npoint, float* temp, int32_t* out, void* stream_) {
    REART_ENTRY();
    if (B < 0 || N < 0 || npoint < 0 || !fits_int(N)) return REART_ERR_INVALID_ARG;
    if (B == 0 || npoint == 0) return REART_OK;
    if (!xyz || !out || N == 0) return REART_ERR_INVALID_ARG;
    // small clouds: the register kernel (temp unused); larger ones: running distances in the caller's temp [B,N]
    if (N <= 32768) return launch_fps(xyz, B, N, npoint, out, static_cast<cudaStream_t>(stream_));
    if (!temp) return REART_ERR_WORKSPACE;
    return launch_fps_large(xyz, B, N, npoint, temp, out, static_cast<cudaStream_t>(stream_));
}

int reart_ball_query(const float* new_xyz, const float* xyz, int64_t B, int64_t N, int64_t m, float radius,
                     int nsample, int32_t* idx, void* stream_) {
    REART_ENTRY();
    if (B < 0 || N < 0 || m < 0 || nsample < 0 || !fits_int(N) || !fits_int(m)) return REART_ERR_INVALID_ARG;
    if (B == 0 || m == 0 || nsample == 0) return REART_OK;
    if (!new_xyz || !idx || (N > 0 && !xyz)) return REART_ERR_INVALID_ARG;
    return launch_ball_query(new_xyz, xyz, B, N, m, radius, nsample, idx, static_cast<cudaStream_t>(stream_));
}

int reart_allreduce_oneshot(const uint64_t* peer_base, int rank, int world, int64_t n, int64_t n_pad, uint32_t* epoch,
                            float* data, void* stream_) {
    REART_ENTRY();
    if (world < 1 || rank < 0 || rank >= world || n < 0 || n_pad < n) return REART_ERR_INVALID_ARG;
    if (n == 0 || world == 1) return REART_OK;
    if (!peer_base || !epoch || !data) return REART_ERR_INVALID_ARG;
    return launch_allreduce_oneshot(reinterpret_cast<const unsigned long long*>(peer_base), rank, world, n, n_pad,
                                    epoch, data, static_cast<cudaStream_t>(stream_));
}

int reart_fp32_probe(int variant, int iters, int blocks, const float* scratch_in, float* scratch_out, double* ms,
                     double* ops_per_thread, void* stream_) {
    REART_ENTRY();
    return launch_probe(variant, iters, blocks, scratch_in, scratch_out, ms, ops_per_thread,
                        static_cast<cudaStream_t>(stream_));
}

}  // extern "C"
