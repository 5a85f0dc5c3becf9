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

// ------------------------------------------------------------------------------------------------
// The convolution AFTER the folded first layer aggregates H1 = act(a u^T + c v^T + b) — rows that are a
// function of two scalars per node.  Z = A2_hat H1 is therefore computed WITHOUT gathering feature rows:
// per edge the kernel fetches (a, c) of the source (8 bytes instead of 4 F), rebuilds the row in registers
// (2 FMA + one ex2 per element) and accumulates.  The gather of [N, F] rows, the dominant cost of a
// normalised aggregation (L2 -> SM fabric bound), becomes MUFU work: F ex2 per edge.
// Warp = 32 consecutive rows, lanes = VEC consecutive features each (F = 32 VEC); (col, val, a, c) of the next
// 32 edges are prefetched lane-parallel and broadcast with shuffles; rows are closed in order.
// Backward: dL/d(u, v, b) = sum_r dZ[r,:] * sum_{e in row r} val_e (a_s, c_s, 1) act'(pre_s) — the same walk,
// three accumulators per feature, one read of dZ per ROW; per-block partials, fixed-order reduction.
// ------------------------------------------------------------------------------------------------
constexpr int kR1RowsPerWarp = 32;
constexpr int kR1Unroll = 4;                 // edges per inner step: independent FMA / ex2 chains

template <int VEC>
__device__ __forceinline__ void ldvec(float (&r)[VEC], const float *p) {
    if constexpr (VEC == 1) { r[0] = __ldg(p); }
    else if constexpr (VEC == 2) { const float2 t = __ldg(reinterpret_cast<const float2 *>(p)); r[0] = t.x; r[1] = t.y; }
    else { const float4 t = __ldg(reinterpret_cast<const float4 *>(p)); r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w; }
}

template <int VEC>
__device__ __forceinline__ void stvec(float *p, const float (&r)[VEC]) {
    if constexpr (VEC == 1) { *p = r[0]; }
    else if constexpr (VEC == 2) { *reinterpret_cast<float2 *>(p) = make_float2(r[0], r[1]); }
    else { *reinterpret_cast<float4 *>(p) = make_float4(r[0], r[1], r[2], r[3]); }
}

// BWD == false: y[r,:] = sum_e val_e act(a_s u + c_s v + b)
// BWD == true : partial[block] = sum over the block's rows of t[r,:] * sum_e val_e (1, a_s, c_s) act'(a_s u + c_s v + b)
template <int VEC, bool BWD>
__global__ void __launch_bounds__(256)
rank1_aggregate_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                       const float *__restrict__ val, const float *__restrict__ a, const float *__restrict__ c,
                       const float *__restrict__ u, const float *__restrict__ v, const float *__restrict__ bias,
                       int32_t num_rows, int act, float *__restrict__ y, int64_t ldy,
                       const float *__restrict__ t, int64_t ldt, float *__restrict__ partial) {
    constexpr int F = 32 * VEC;
    __shared__ float red[BWD ? 8 * 3 * F : 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * kR1RowsPerWarp;
    float s0[VEC], s1[VEC], s2[VEC];                         // BWD: running column sums of this warp
#pragma unroll
    for (int k = 0; k < VEC; ++k) s0[k] = s1[k] = s2[k] = 0.f;
    if (r0 < num_rows) {
        const int nrows = (int)min((int64_t)kR1RowsPerWarp, (int64_t)num_rows - r0);
        const int64_t e_begin = rowptr[r0];
        const int my_end = (int)(rowptr[r0 + min(lane, nrows - 1) + 1] - e_begin);
        const int n_edges = __shfl_sync(0xffffffffu, my_end, nrows - 1);
        col += e_begin;
        val += e_begin;
        float uu[VEC], vv[VEC], bb[VEC];
        ldvec<VEC>(uu, u + lane * VEC);
        ldvec<VEC>(vv, v + lane * VEC);
#pragma unroll
        for (int k = 0; k < VEC; ++k) bb[k] = 0.f;
        if (bias) ldvec<VEC>(bb, bias + lane * VEC);
        int cur = 0;
        int cur_end = __shfl_sync(0xffffffffu, my_end, 0);
        float q0[VEC], q1[VEC], q2[VEC];
#pragma unroll
        for (int k = 0; k < VEC; ++k) q0[k] = q1[k] = q2[k] = 0.f;

        auto close_row = [&]() {
            if constexpr (!BWD) {
                stvec<VEC>(y + (r0 + cur) * ldy + lane * VEC, q0);
            } else {
                float tt[VEC];
                ldvec<VEC>(tt, t + (r0 + cur) * ldt + lane * VEC);
#pragma unroll
                for (int k = 0; k < VEC; ++k) {
                    s0[k] = fmaf(tt[k], q0[k], s0[k]);
                    s1[k] = fmaf(tt[k], q1[k], s1[k]);
                    s2[k] = fmaf(tt[k], q2[k], s2[k]);
                }
            }
#pragma unroll
            for (int k = 0; k < VEC; ++k) q0[k] = q1[k] = q2[k] = 0.f;
            ++cur;
            cur_end = __shfl_sync(0xffffffffu, my_end, cur & 31);
        };

        auto edge = [&](float we, float as, float cs, int k) {
            const float pre = fmaf(as, uu[k], fmaf(cs, vv[k], bb[k]));
            if constexpr (!BWD) {
                const float h = (act == PANGNN_ACT_ELU && pre <= 0.f) ? __expf(pre) - 1.f : pre;
                q0[k] = fmaf(we, h, q0[k]);
            } else {
                const float d = (act == PANGNN_ACT_ELU && pre <= 0.f) ? __expf(pre) : 1.f;
                const float wd = we * d;
                q0[k] += wd;
                q1[k] = fmaf(as, wd, q1[k]);
                q2[k] = fmaf(cs, wd, q2[k]);
            }
        };

        float w_n = 0.f, a_n = 0.f, c_n = 0.f;
        if (lane < n_edges) {
            const int32_t s = col[lane];
            w_n = val[lane]; a_n = a[s]; c_n = c[s];
        }
        for (int base = 0; base < n_edges; base += 32) {
            const float w_c = w_n, a_c = a_n, c_c = c_n;
            const int nb = base + 32 + lane;
            if (nb < n_edges) {                                 // prefetch the next 32 edges, lane-parallel
                const int32_t s = col[nb];
                w_n = val[nb]; a_n = a[s]; c_n = c[s];
            }
            const int cnt = min(32, n_edges - base);
            for (int j0 = 0; j0 < cnt; j0 += kR1Unroll) {
                float we[kR1Unroll], as[kR1Unroll], cs[kR1Unroll];
#pragma unroll
                for (int q = 0; q < kR1Unroll; ++q) {
                    we[q] = __shfl_sync(0xffffffffu, w_c, (j0 + q) & 31);
                    as[q] = __shfl_sync(0xffffffffu, a_c, (j0 + q) & 31);
                    cs[q] = __shfl_sync(0xffffffffu, c_c, (j0 + q) & 31);
                }
                const int e0 = base + j0;
                if (e0 + kR1Unroll <= cur_end) {                // whole group inside the open row: independent chains
#pragma unroll
                    for (int q = 0; q < kR1Unroll; ++q)
#pragma unroll
                        for (int k = 0; k < VEC; ++k) edge(we[q], as[q], cs[q], k);
                } else {
#pragma unroll
                    for (int q = 0; q < kR1Unroll; ++q) {
                        if (e0 + q < n_edges) {                 // warp-uniform
                            while (e0 + q >= cur_end) close_row();   // rows ending before this edge (incl. empty ones)
#pragma unroll
                            for (int k = 0; k < VEC; ++k) edge(we[q], as[q], cs[q], k);
                        }
                    }
                }
            }
        }
        while (cur < nrows) close_row();
    }
    if constexpr (BWD) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            red[(warp * 3 + 0) * F + lane * VEC + k] = s0[k];
            red[(warp * 3 + 1) * F + lane * VEC + k] = s1[k];
            red[(warp * 3 + 2) * F + lane * VEC + k] = s2[k];
        }
        __syncthreads();
        for (int i = threadIdx.x; i < 3 * F; i += blockDim.x) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < 8; ++w) s += red[w * 3 * F + i];
            partial[(int64_t)blockIdx.x * 3 * F + i] = s;
        }
    }
}

static int64_t r1_agg_blocks(int64_t num_rows) {
    const int64_t warps = (num_rows + kR1RowsPerWarp - 1) / kR1RowsPerWarp;
    return (warps * 32 + 255) / 256;
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

int pangnn_rank1_aggregate(const int64_t *rowptr, const int32_t *col, const float *val, const float *a, const float *c,
                           const float *u, const float *v, const float *bias, int32_t num_rows, int32_t feat, int act,
                           float *y, int64_t ldy, void *stream) {
    if (num_rows <= 0) return PANGNN_OK;
    PANGNN_REQUIRE(rowptr && a && c && u && v && y, "null pointer");       // col / val may be NULL without edges
    PANGNN_REQUIRE(feat == 32 || feat == 64 || feat == 128, "feat must be 32, 64 or 128");
    PANGNN_REQUIRE(ldy % 4 == 0 && ldy >= feat && (uintptr_t)y % 16 == 0 && (uintptr_t)u % 16 == 0 &&
                       (uintptr_t)v % 16 == 0 && (!bias || (uintptr_t)bias % 16 == 0), "alignment");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)r1_agg_blocks(num_rows);
#define R1LAUNCH(VEC)                                                                                          \
    rank1_aggregate_kernel<VEC, false><<<blocks, 256, 0, st>>>(rowptr, col, val, a, c, u, v, bias, num_rows, act, y, \
                                                               ldy, nullptr, 0, nullptr)
    if (feat == 128) R1LAUNCH(4);
    else if (feat == 64) R1LAUNCH(2);
    else R1LAUNCH(1);
#undef R1LAUNCH
    PANGNN_CHECK_LAUNCH("rank1_aggregate");
    return PANGNN_OK;
}

size_t pangnn_rank1_aggregate_bwd_workspace_bytes(int64_t num_rows, int32_t feat) {
    return (size_t)r1_agg_blocks(num_rows) * 3 * feat * sizeof(float) + 256;
}

int pangnn_rank1_aggregate_bwd(const int64_t *rowptr, const int32_t *col, const float *val, const float *a,
                               const float *c, const float *u, const float *v, const float *bias, int32_t num_rows,
                               int32_t feat, int act, const float *dz, int64_t lddz, float *sums, void *ws,
                               size_t ws_bytes, void *stream) {
    PANGNN_REQUIRE(rowptr && a && c && u && v && sums && ws, "null pointer");
    PANGNN_REQUIRE(feat == 32 || feat == 64 || feat == 128, "feat must be 32, 64 or 128");
    if (ws_bytes < pangnn_rank1_aggregate_bwd_workspace_bytes(num_rows, feat)) {
        set_error("rank1_aggregate_bwd: workspace too small");
        return PANGNN_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (num_rows <= 0) return check_cuda(cudaMemsetAsync(sums, 0, 3 * feat * sizeof(float), st), "memset");
    PANGNN_REQUIRE(dz && lddz % 4 == 0 && lddz >= feat && (uintptr_t)dz % 16 == 0, "dz alignment");
    const int64_t nb = r1_agg_blocks(num_rows);
    float *partial = static_cast<float *>(ws);
#define R1LAUNCH(VEC)                                                                                          \
    rank1_aggregate_kernel<VEC, true><<<(unsigned)nb, 256, 0, st>>>(rowptr, col, val, a, c, u, v, bias, num_rows, act, \
                                                                    nullptr, 0, dz, lddz, partial)
    if (feat == 128) R1LAUNCH(4);
    else if (feat == 64) R1LAUNCH(2);
    else R1LAUNCH(1);
#undef R1LAUNCH
    PANGNN_CHECK_LAUNCH("rank1_aggregate_bwd");
    return reduce_partials(partial, nb, 3 * feat, 3 * feat, sums, st);
}

}  // extern "C"
