// C ABI of the fused edge scorer (argument checks, workspace carving, second-stage reductions) and
// the cosine / dot decoders.  The tile kernel itself — endpoint gather, 3-layer MLP, BCE loss and the
// whole backward on the tcgen05 tensor cores — is edge_scorer_tc.cu; see its header for the design.
// Replaces src/gnn.py:171-180,202-207, pangnn.py:98,203 and their autograd backward (pangnn.py:207).
// The per-node gradients are sorted-segment reductions of da1 (pangnn_gcn_aggregate with val = NULL
// over the by-source / by-destination CSR of the scored edges) — no atomics anywhere.
#include "edge_scorer.cuh"

namespace pangnn {

int reduce_partials(const float *partial, int64_t nblocks, int32_t width, int32_t stride, float *out,
                    cudaStream_t st);

constexpr int NG = kScNG;
constexpr int NGP = kScNGP;

__global__ void reduce_loss_kernel(const double *__restrict__ partial, int n, double *__restrict__ out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < n; ++i) s += partial[i];
        *out += s;
    }
}

// cosine similarity (F.cosine_similarity, eps = 1e-8 on each norm) / row-wise dot, warp per edge
__global__ void __launch_bounds__(256)
edge_pair_score_kernel(const float *__restrict__ h, int64_t ldh, int32_t feat,
                       const int32_t *__restrict__ src, const int32_t *__restrict__ dst, int64_t E,
                       int mode, float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (e >= E) return;
    const float *a = h + (int64_t)src[e] * ldh, *b = h + (int64_t)dst[e] * ldh;
    float ab = 0.f, aa = 0.f, bb = 0.f;
    for (int f = lane; f < feat; f += 32) {
        const float x = a[f], yv = b[f];
        ab = fmaf(x, yv, ab); aa = fmaf(x, x, aa); bb = fmaf(yv, yv, bb);
    }
    ab = warp_sum(ab); aa = warp_sum(aa); bb = warp_sum(bb);
    if (lane == 0) {
        if (mode == 0) {
            const float eps = 1e-8f;
            out[e] = ab / (fmaxf(sqrtf(aa), eps) * fmaxf(sqrtf(bb), eps));
        } else {
            out[e] = ab;
        }
    }
}

// ---- backward of the cosine / dot decoders (src/gnn.py:202-207 under autograd, pangnn.py:207) -------------
// With c_e the forward value, na = max(|h_s|, eps), nb = max(|h_d|, eps), and the norm differentiated as torch's
// F.cosine_similarity does (clamped value, unclamped derivative h / |h|; 0 for an all-zero row):
//   d/dh_s = dz_e (h_d / (na nb) - c_e h_s / (na |h_s|)),   d/dh_d = dz_e (h_s / (na nb) - c_e h_d / (nb |h_d|))
// so the node gradient is TWO weighted aggregations over the scored-edge graph plus a diagonal term,
//   dh = A_src(alpha) h + A_dst(alpha) h - diag(beta) h,   alpha_e = dz_e / (na nb),
//   beta_n = sum_{e: src = n} dz_e c_e / (na |h_s|) + sum_{e: dst = n} dz_e c_e / (nb |h_d|)
// (dot: alpha_e = dz_e, beta = 0) — no per-edge [E, F] gradient rows are ever materialised; the aggregations
// run on the streaming gather kernel of the convolutions (gcn.cu), the reduction order is the CSR order.
__global__ void __launch_bounds__(256)
row_norm_kernel(const float *__restrict__ h, int64_t ldh, int32_t feat, int32_t N, float *__restrict__ nrm) {
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= N) return;
    const float *a = h + r * ldh;
    float s = 0.f;
    for (int f = lane; f < feat; f += 32) s = fmaf(a[f], a[f], s);
    s = warp_sum(s);
    if (lane == 0) nrm[r] = sqrtf(s);                    // unclamped: the eps clamp is applied by the user
}

// warp per CSR row r: val[p] = alpha of slot p, diag[r] (+)= the row's beta sum (fixed lane-strided order)
__global__ void __launch_bounds__(256)
pair_coef_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col, const uint32_t *__restrict__ perm,
                 const float *__restrict__ dz, const float *__restrict__ out, const float *__restrict__ nrm,
                 int mode, int32_t N, int accumulate, float *__restrict__ val, float *__restrict__ diag) {
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= N) return;
    const int64_t b = rowptr[r], e = rowptr[r + 1];
    const float eps = 1e-8f;
    const float rr = mode == 0 ? nrm[r] : 1.f;           // |h_r|
    const float nr = fmaxf(rr, eps);
    float beta = 0.f;
    for (int64_t p = b + lane; p < e; p += 32) {
        const uint32_t ed = perm[p];
        const float g = dz[ed];
        if (mode == 0) {
            val[p] = g / (nr * fmaxf(nrm[col[p]], eps));
            if (rr > 0.f) beta += g * out[ed] / (nr * rr);
        } else {
            val[p] = g;
        }
    }
    beta = warp_sum(beta);
    if (lane == 0) diag[r] = accumulate ? diag[r] + beta : beta;
}

// dh += t - diag * h   (rows of width feat; float4 lanes)
__global__ void __launch_bounds__(256)
pair_combine_kernel(const float *__restrict__ t, const float *__restrict__ diag, const float *__restrict__ h, int64_t ldh,
                    int32_t feat, int64_t N, float *__restrict__ dh) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int f4 = feat >> 2;
    if (i >= N * f4) return;
    const int64_t r = i / f4;
    const int c = (int)(i % f4) * 4;
    const float d = diag[r];
    const float4 tv = *reinterpret_cast<const float4 *>(t + r * feat + c);
    const float4 hv = *reinterpret_cast<const float4 *>(h + r * ldh + c);
    float4 o = *reinterpret_cast<float4 *>(dh + r * feat + c);
    o.x += tv.x - d * hv.x; o.y += tv.y - d * hv.y; o.z += tv.z - d * hv.z; o.w += tv.w - d * hv.w;
    *reinterpret_cast<float4 *>(dh + r * feat + c) = o;
}

// doubles (per-CTA loss partials) live after the float partials
constexpr size_t kLossOff = (size_t)kNumSMs * 2 * NGP * sizeof(float);

}  // namespace pangnn

using namespace pangnn;

extern "C" {

size_t pangnn_edge_score_workspace_bytes(int64_t E) {
    (void)E;
    return kLossOff + (size_t)kNumSMs * 4 * sizeof(double) + 1024;
}

int pangnn_edge_score_fwd(const float *pq, const int32_t *src, const int32_t *dst, const float *skip,
                          const float *w1c, const float *b1, const float *w2, const float *b2,
                          const float *w3, const float *b3, int64_t E, const float *y,
                          float pos_weight, float *logits, double *loss_sum, void *ws,
                          size_t ws_bytes, void *stream) {
    PANGNN_REQUIRE(E >= 0, "negative edge count");
    if (E == 0) return PANGNN_OK;
    PANGNN_REQUIRE(pq && src && dst && b1 && w2 && b2 && w3 && b3, "null pointer");
    PANGNN_REQUIRE(!skip || w1c, "skip feature needs w1c");
    PANGNN_REQUIRE(!loss_sum || (y && ws), "loss needs labels and a workspace");
    PANGNN_REQUIRE((uintptr_t)pq % 16 == 0, "pq must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (loss_sum && ws_bytes < pangnn_edge_score_workspace_bytes(E)) {
        set_error("edge_score_fwd: workspace too small");
        return PANGNN_EWORKSPACE;
    }
    ScorerArgs a{};
    a.pq = pq; a.src = src; a.dst = dst; a.skip = skip; a.w1c = w1c; a.b1 = b1; a.w2 = w2; a.b2 = b2;
    a.w3 = w3; a.b3 = b3; a.E = E; a.y = loss_sum ? y : nullptr; a.pos_weight = pos_weight;
    a.logits = logits;
    a.loss_partial = loss_sum ? reinterpret_cast<double *>(static_cast<char *>(ws) + kLossOff) : nullptr;
    int grid = 0;
    int rc = launch_edge_score_tc(a, false, &grid, st);
    if (rc) return rc;
    if (loss_sum) {
        reduce_loss_kernel<<<1, 32, 0, st>>>(a.loss_partial, grid, loss_sum);
        PANGNN_CHECK_LAUNCH("reduce_loss");
    }
    return PANGNN_OK;
}

int pangnn_edge_score_predict(const float *pq, const int32_t *src, const int32_t *dst, const float *skip,
                              const float *w1c, const float *b1, const float *w2, const float *b2,
                              const float *w3, const float *b3, int64_t E, float threshold, float *logits,
                              float *prob, int32_t *pred, void *stream) {
    PANGNN_REQUIRE(E >= 0, "negative edge count");
    if (E == 0) return PANGNN_OK;
    PANGNN_REQUIRE(pq && src && dst && b1 && w2 && b2 && w3 && b3, "null pointer");
    PANGNN_REQUIRE(!skip || w1c, "skip feature needs w1c");
    PANGNN_REQUIRE((uintptr_t)pq % 16 == 0, "pq must be 16-byte aligned");
    ScorerArgs a{};
    a.pq = pq; a.src = src; a.dst = dst; a.skip = skip; a.w1c = w1c; a.b1 = b1; a.w2 = w2; a.b2 = b2;
    a.w3 = w3; a.b3 = b3; a.E = E; a.logits = logits; a.prob = prob; a.pred = pred; a.threshold = threshold;
    int grid = 0;
    return launch_edge_score_tc(a, false, &grid, (cudaStream_t)stream);
}

int pangnn_edge_score_bwd(const float *pq, const int32_t *src, const int32_t *dst, const float *skip,
                          const float *w1c, const float *b1, const float *w2, const float *b2,
                          const float *w3, const float *b3, int64_t E, const float *dlogits,
                          const float *y, float pos_weight, float scale, float *da1, float *grads,
                          float *logits, double *loss_sum, void *ws, size_t ws_bytes, void *stream) {
    PANGNN_REQUIRE(E >= 0 && grads, "bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    if (E == 0) return check_cuda(cudaMemsetAsync(grads, 0, NG * sizeof(float), st), "memset");
    PANGNN_REQUIRE(pq && src && dst && b1 && w2 && b2 && w3 && b3 && da1 && ws, "null pointer");
    PANGNN_REQUIRE(dlogits || y, "need dlogits or labels");
    PANGNN_REQUIRE(!skip || w1c, "skip feature needs w1c");
    PANGNN_REQUIRE((uintptr_t)pq % 16 == 0 && (uintptr_t)da1 % 16 == 0, "pointers must be 16-byte aligned");
    if (ws_bytes < pangnn_edge_score_workspace_bytes(E)) {
        set_error("edge_score_bwd: workspace too small");
        return PANGNN_EWORKSPACE;
    }
    ScorerArgs a{};
    a.pq = pq; a.src = src; a.dst = dst; a.skip = skip; a.w1c = w1c; a.b1 = b1; a.w2 = w2; a.b2 = b2;
    a.w3 = w3; a.b3 = b3; a.E = E; a.y = y; a.dlogits = dlogits; a.pos_weight = pos_weight;
    a.scale = scale; a.da1 = da1; a.partial = static_cast<float *>(ws);
    a.logits = logits;
    PANGNN_REQUIRE(!loss_sum || y, "loss needs labels");
    a.loss_partial = loss_sum ? reinterpret_cast<double *>(static_cast<char *>(ws) + kLossOff) : nullptr;
    int grid = 0;
    int rc = launch_edge_score_tc(a, true, &grid, st);
    if (rc) return rc;
    if (loss_sum) {
        reduce_loss_kernel<<<1, 32, 0, st>>>(a.loss_partial, grid, loss_sum);
        PANGNN_CHECK_LAUNCH("reduce_loss");
    }
    return reduce_partials(a.partial, grid, NG, NGP, grads, st);
}

int pangnn_edge_pair_score(const float *h, int64_t ldh, int32_t feat, const int32_t *src,
                           const int32_t *dst, int64_t E, int mode, float *out, void *stream) {
    PANGNN_REQUIRE(E >= 0, "negative edge count");
    if (E == 0) return PANGNN_OK;
    PANGNN_REQUIRE(h && src && dst && out && feat > 0, "null pointer");
    const unsigned blocks = (unsigned)((E * 32 + 255) / 256);
    edge_pair_score_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(h, ldh, feat, src, dst, E, mode, out);
    PANGNN_CHECK_LAUNCH("edge_pair_score");
    return PANGNN_OK;
}

size_t pangnn_edge_pair_score_bwd_workspace_bytes(int64_t E, int32_t N, int32_t feat) {
    return align_up((size_t)E * 4, 256) + 2 * align_up((size_t)N * 4, 256) + align_up((size_t)N * feat * 4, 256) + 256;
}

int pangnn_edge_pair_score_bwd(const float *h, int64_t ldh, int32_t feat, int32_t N, int64_t E,
                               const int64_t *rowptr_src, const int32_t *col_src, const uint32_t *perm_src,
                               const int64_t *rowptr_dst, const int32_t *col_dst, const uint32_t *perm_dst,
                               const float *dz, const float *out, int mode, float *dh, void *ws, size_t ws_bytes,
                               void *stream) {
    PANGNN_REQUIRE(E >= 0 && N >= 0 && feat > 0 && feat % 4 == 0, "bad arguments (feat must be a multiple of 4)");
    if (N == 0) return PANGNN_OK;
    PANGNN_REQUIRE(h && dh && ws && rowptr_src && rowptr_dst, "null pointer");
    PANGNN_REQUIRE(E == 0 || (col_src && perm_src && col_dst && perm_dst && dz && out), "null pointer");
    PANGNN_REQUIRE(ldh % 4 == 0 && (uintptr_t)h % 16 == 0 && (uintptr_t)dh % 16 == 0, "rows must be 16-byte aligned");
    if (ws_bytes < pangnn_edge_pair_score_bwd_workspace_bytes(E, N, feat)) {
        set_error("edge_pair_score_bwd: workspace too small");
        return PANGNN_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    Workspace w(ws, ws_bytes);
    float *val = w.take<float>((size_t)E), *nrm = w.take<float>((size_t)N), *diag = w.take<float>((size_t)N);
    float *tmp = w.take<float>((size_t)N * feat);
    const unsigned wblocks = (unsigned)(((int64_t)N * 32 + 255) / 256);
    if (mode == 0) {
        row_norm_kernel<<<wblocks, 256, 0, st>>>(h, ldh, feat, N, nrm);
        PANGNN_CHECK_LAUNCH("row_norm");
    }
    pair_coef_kernel<<<wblocks, 256, 0, st>>>(rowptr_src, col_src, perm_src, dz, out, nrm, mode, N, 0, val, diag);
    PANGNN_CHECK_LAUNCH("pair_coef(src)");
    int rc = pangnn_gcn_aggregate(rowptr_src, col_src, val, h, ldh, N, feat, nullptr, PANGNN_ACT_NONE, dh, feat, stream);
    if (rc) return rc;
    pair_coef_kernel<<<wblocks, 256, 0, st>>>(rowptr_dst, col_dst, perm_dst, dz, out, nrm, mode, N, 1, val, diag);
    PANGNN_CHECK_LAUNCH("pair_coef(dst)");
    rc = pangnn_gcn_aggregate(rowptr_dst, col_dst, val, h, ldh, N, feat, nullptr, PANGNN_ACT_NONE, tmp, feat, stream);
    if (rc) return rc;
    const int64_t n4 = (int64_t)N * (feat / 4);
    pair_combine_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(tmp, diag, h, ldh, feat, N, dh);
    PANGNN_CHECK_LAUNCH("pair_combine");
    return PANGNN_OK;
}

}  // extern "C"
