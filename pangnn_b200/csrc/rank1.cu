// Embedding Linear(1, D) + first GCNConv as ONE rank-2 update (src/gnn.py:97,125 followed by :129 / :135 /
// :147).  The node features of the reference are a single scalar per gene (x = ones [N, 1]), so the embedding
// E0 = x w_e^T + 1 b_e^T has rank 2 and the first convolution is linear in it:
//     A_hat (E0 W^T) + b  =  (A_hat x) (W w_e)^T + (A_hat 1) (W b_e)^T + b  =  a u^T + c v^T + b
// with two N-vectors a = A_hat x, c = A_hat 1 (one SpMV pass over the CSR; they depend on the graph, the edge
// weights and x only, so they are cached with gcn_norm) and two F-vectors u = W w_e, v = W b_e.  The layer is
// then one streaming write of [N, F] forward and one streaming read of dY, Y backward (three weighted column
// sums: db = sum g, du = sum a g, dv = sum c g; dW = du w_e^T + dv b_e^T, dw_e = W^T du, db_e = W^T dv) —
// instead of an [N, D] embedding pass, a width-D aggregation forward and backward, and three N x D x F GEMMs.
#include "common.cuh"

namespace pangnn {

int reduce_partials(const float *partial, int64_t nblocks, int32_t width, int32_t stride, float *out,
                    cudaStream_t st);

// a[r] = sum_e val_e x[col_e], c[r] = sum_e val_e   (warp per row, fp64 accumulate, lanes strided over the row)
__global__ void __launch_bounds__(256)
csr_spmv2_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col, const float *__restrict__ val,
                 const float *__restrict__ x, int32_t N, float *__restrict__ ax, float *__restrict__ a1) {
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= N) return;
    const int64_t b = rowptr[row], e = rowptr[row + 1];
    double sx = 0.0, s1 = 0.0;
    for (int64_t i = b + lane; i < e; i += 32) {
        const double v = (double)val[i];
        s1 += v;
        sx += x ? v * (double)x[col[i]] : v;
    }
    sx = warp_sum(sx);
    s1 = warp_sum(s1);
    if (lane == 0) {
        ax[row] = (float)sx;
        a1[row] = (float)s1;
    }
}

__device__ __forceinline__ float act_apply(float x, int act) {
    return (act == PANGNN_ACT_ELU && x <= 0.f) ? expm1f(x) : x;
}

// y[r, :] = act(a[r] u + c[r] v + b): one float4 per thread
__global__ void __launch_bounds__(256)
rank1_affine_act_kernel(const float *__restrict__ a, const float *__restrict__ c, const float *__restrict__ u,
                        const float *__restrict__ v, const float *__restrict__ bias, int64_t num_rows, int32_t fq,
                        int act, float *__restrict__ y, int64_t ldy) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= num_rows * fq) return;
    const int64_t r = i / fq;
    const int t = (int)(i % fq);
    const float ar = a[r], cr = c[r];
    const float4 uu = __ldg(reinterpret_cast<const float4 *>(u) + t), vv = __ldg(reinterpret_cast<const float4 *>(v) + t);
    float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias) bb = __ldg(reinterpret_cast<const float4 *>(bias) + t);
    float4 o;
    o.x = act_apply(fmaf(ar, uu.x, fmaf(cr, vv.x, bb.x)), act);
    o.y = act_apply(fmaf(ar, uu.y, fmaf(cr, vv.y, bb.y)), act);
    o.z = act_apply(fmaf(ar, uu.z, fmaf(cr, vv.z, bb.z)), act);
    o.w = act_apply(fmaf(ar, uu.w, fmaf(cr, vv.w, bb.w)), act);
    reinterpret_cast<float4 *>(y + r * ldy)[t] = o;
}

constexpr int kR1RowsPerChunk = 64;
constexpr int kR1MaxBlocks = kNumSMs * 8;

// g = dy * act'(y); partial[b] = (sum g | sum a g | sum c g) over the rows of block b  ([3][feat])
__global__ void __launch_bounds__(256)
rank1_bwd_kernel(const float *__restrict__ dy, const float *__restrict__ yv, const float *__restrict__ a,
                 const float *__restrict__ c, int64_t num_rows, int32_t feat, int act, float *__restrict__ partial) {
    extern __shared__ float4 red[];                        // [TY][3][feat/4]
    const int fq = feat / 4;
    const int tx = threadIdx.x % fq, ty = threadIdx.x / fq;
    const int TY = blockDim.x / fq;
    const int64_t nchunks = (num_rows + kR1RowsPerChunk - 1) / kR1RowsPerChunk;
    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0, s2 = s0;
    if (ty < TY) {
        for (int64_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
            const int64_t r0 = chunk * kR1RowsPerChunk;
            const int64_t r1 = min(r0 + (int64_t)kR1RowsPerChunk, num_rows);
            for (int64_t r = r0 + ty; r < r1; r += TY) {
                float4 d = ld_stream_f4(dy + r * feat + tx * 4);
                if (act == PANGNN_ACT_ELU) {
                    const float4 o = ld_stream_f4(yv + r * feat + tx * 4);
                    d.x *= o.x > 0.f ? 1.f : o.x + 1.f;
                    d.y *= o.y > 0.f ? 1.f : o.y + 1.f;
                    d.z *= o.z > 0.f ? 1.f : o.z + 1.f;
                    d.w *= o.w > 0.f ? 1.f : o.w + 1.f;
                }
                const float ar = a[r], cr = c[r];
                s0.x += d.x; s0.y += d.y; s0.z += d.z; s0.w += d.w;
                s1.x = fmaf(ar, d.x, s1.x); s1.y = fmaf(ar, d.y, s1.y); s1.z = fmaf(ar, d.z, s1.z); s1.w = fmaf(ar, d.w, s1.w);
                s2.x = fmaf(cr, d.x, s2.x); s2.y = fmaf(cr, d.y, s2.y); s2.z = fmaf(cr, d.z, s2.z); s2.w = fmaf(cr, d.w, s2.w);
            }
        }
        red[(ty * 3 + 0) * fq + tx] = s0;
        red[(ty * 3 + 1) * fq + tx] = s1;
        red[(ty * 3 + 2) * fq + tx] = s2;
    }
    __syncthreads();
    if (ty == 0) {
        for (int k = 0; k < 3; ++k) {
            float4 s = red[k * fq + tx];
            for (int t = 1; t < TY; ++t) {
                const float4 o = red[(t * 3 + k) * fq + tx];
                s.x += o.x; s.y += o.y; s.z += o.z; s.w += o.w;
            }
            reinterpret_cast<float4 *>(partial + ((int64_t)blockIdx.x * 3 + k) * feat)[tx] = s;
        }
    }
}

static int64_t r1_blocks(int64_t num_rows) {
    const int64_t nchunks = (num_rows + kR1RowsPerChunk - 1) / kR1RowsPerChunk;
    return nchunks < 1 ? 1 : (nchunks < kR1MaxBlocks ? nchunks : kR1MaxBlocks);
}

}  // namespace pangnn

using namespace pangnn;

extern "C" {

int pangnn_csr_spmv2(const int64_t *rowptr, const int32_t *col, const float *val, const float *x, int32_t num_rows,
                     float *ax, float *a1, void *stream) {
    if (num_rows <= 0) return PANGNN_OK;
    PANGNN_REQUIRE(rowptr && ax && a1, "null pointer");     // col / val may be NULL for an edgeless graph
    const unsigned blocks = (unsigned)(((int64_t)num_rows * 32 + 255) / 256);
    csr_spmv2_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rowptr, col, val, x, num_rows, ax, a1);
    PANGNN_CHECK_LAUNCH("csr_spmv2");
    return PANGNN_OK;
}

int pangnn_rank1_affine_act(const float *a, const float *c, const float *u, const float *v, const float *bias,
                            int64_t num_rows, int32_t feat, int act, float *y, int64_t ldy, void *stream) {
    if (num_rows <= 0) return PANGNN_OK;
    PANGNN_REQUIRE(a && c && u && v && y, "null pointer");
    PANGNN_REQUIRE(feat > 0 && feat % 4 == 0 && ldy % 4 == 0 && ldy >= feat, "feat / ldy must be multiples of 4");
    PANGNN_REQUIRE((uintptr_t)u % 16 == 0 && (uintptr_t)v % 16 == 0 && (uintptr_t)y % 16 == 0 &&
                       (!bias || (uintptr_t)bias % 16 == 0), "pointers must be 16-byte aligned");
    const int64_t total = num_rows * (feat / 4);
    rank1_affine_act_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        a, c, u, v, bias, num_rows, feat / 4, act, y, ldy);
    PANGNN_CHECK_LAUNCH("rank1_affine_act");
    return PANGNN_OK;
}

size_t pangnn_rank1_bwd_workspace_bytes(int64_t num_rows, int32_t feat) {
    return (size_t)r1_blocks(num_rows) * 3 * feat * sizeof(float) + 256;
}

int pangnn_rank1_bwd(const float *dy, const float *yv, const float *a, const float *c, int64_t num_rows, int32_t feat,
                     int act, float *sums, void *ws, size_t ws_bytes, void *stream) {
    PANGNN_REQUIRE(sums && ws, "null pointer");
    PANGNN_REQUIRE(feat > 0 && feat % 4 == 0 && feat <= 256, "feat must be a multiple of 4, <= 256");
    if (ws_bytes < pangnn_rank1_bwd_workspace_bytes(num_rows, feat)) {
        set_error("rank1_bwd: workspace too small");
        return PANGNN_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // zero rows: the inputs are empty tensors, whose data pointer is NULL
    if (num_rows == 0) return check_cuda(cudaMemsetAsync(sums, 0, 3 * feat * sizeof(float), st), "memset");
    PANGNN_REQUIRE(dy && a && c, "null pointer");
    PANGNN_REQUIRE(act == PANGNN_ACT_NONE || yv, "activation output required");
    const int64_t nb = r1_blocks(num_rows);
    const int fq = feat / 4;
    const int TY = 256 / fq;
    float *partial = static_cast<float *>(ws);
    rank1_bwd_kernel<<<(unsigned)nb, 256, (size_t)TY * 3 * fq * sizeof(float4), st>>>(dy, yv, a, c, num_rows, feat, act,
                                                                                     partial);
    PANGNN_CHECK_LAUNCH("rank1_bwd");
    return reduce_partials(partial, nb, 3 * feat, 3 * feat, sums, st);
}

}  // extern "C"
