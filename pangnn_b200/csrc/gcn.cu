// GCN normalisation and the normalised gather-reduce (CSR SpMM) that carries both the forward
// propagate (by-destination CSR) and its backward (transposed CSR).  Replaces
// torch_geometric.nn.GCNConv's gcn_norm + propagate (call sites src/gnn.py:129-165) and the
// autograd scatter/gather pair behind pangnn.py:207.
//
// Roofline: HBM.  Algorithmic bytes per call (SURVEY.md §8d):
//     E*(4 col + 4 val + 4F row) + N*4F (output) + 8(N+1) (rowptr)
// One warp owns one destination row (sorted-segment reduction, no atomics, deterministic order).
// A row of F floats is fetched as F/4 float4 lanes, so a warp keeps 32/(F/4) edges in flight per
// load instruction and UNROLL independent instructions before the first FMA.
#include "common.cuh"

namespace pangnn {

// ------------------------------------------------------------------------------------------------
// gcn_norm
// ------------------------------------------------------------------------------------------------
// deg by destination: warp-per-row sorted-segment sum in fp64, then dis = deg^-1/2 (0 if deg == 0).
__global__ void __launch_bounds__(256)
gcn_deg_kernel(const int64_t *__restrict__ rowptr, const uint32_t *__restrict__ perm,
               const float *__restrict__ w, int32_t N, float *__restrict__ dis) {
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= N) return;
    const int64_t b = rowptr[row], e = rowptr[row + 1];
    double s = 0.0;
    if (w) {
        for (int64_t i = b + lane; i < e; i += 32) s += (double)w[perm[i]];
        s = warp_sum(s);
    } else {
        s = (double)(e - b);
    }
    if (lane == 0) {
        // PyG: deg.pow(-0.5) in fp32, inf -> 0
        const float deg = (float)s;
        dis[row] = deg > 0.f ? 1.0f / sqrtf(deg) : 0.f;
    }
}

// val_e = dis[row] * w_e * dis[col_e] for any CSR ordering of the edge set (row/col roles swap for
// the transposed CSR but the product is symmetric in the two endpoints).
__global__ void __launch_bounds__(256)
gcn_val_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
               const uint32_t *__restrict__ perm, const float *__restrict__ w,
               const float *__restrict__ dis, int32_t N, int rows_are_dst,
               float *__restrict__ val) {
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= N) return;
    const int64_t b = rowptr[row], e = rowptr[row + 1];
    const float dr = dis[row];
    for (int64_t i = b + lane; i < e; i += 32) {
        const float we = w ? w[perm[i]] : 1.0f;
        const float dc = dis[col[i]];
        // same grouping as PyG, (dis[src] * w) * dis[dst]: ((a*w)*b) and ((b*w)*a) can differ
        // in the last ulp, so the source endpoint is multiplied first.
        val[i] = rows_are_dst ? (dc * we) * dr : (dr * we) * dc;
    }
}

// ------------------------------------------------------------------------------------------------
// aggregation
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float elu1(float x) { return x > 0.f ? x : expm1f(x); }

// LPR = lanes per row (F/4 <= LPR, power of two <= 32).  EPW = 32/LPR edges per warp-wide load.
template <int LPR, int UNROLL>
__global__ void __launch_bounds__(256)
gcn_aggregate_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                     const float *__restrict__ val, const float *__restrict__ x, int64_t ldx,
                     int32_t num_rows, int32_t feat, const float *__restrict__ bias, int act,
                     float *__restrict__ y, int64_t ldy) {
    constexpr int EPW = 32 / LPR;
    const int lane = threadIdx.x & 31;
    const int sub = lane / LPR;            // which of the EPW concurrent edges this lane serves
    const int fl = lane % LPR;             // float4 slot inside the row
    const bool active = fl * 4 < feat;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= num_rows) return;
    const int64_t b = rowptr[row], e = rowptr[row + 1];

    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t base = b; base < e; base += 32) {
        // coalesced fetch of up to 32 (col, val) pairs, then broadcast by shuffle
        const int64_t mine = base + lane;
        int32_t c = 0;
        float v = 0.f;
        if (mine < e) {
            c = col[mine];
            v = val ? val[mine] : 1.0f;
        }
        const int cnt = (int)min((int64_t)32, e - base);
        for (int j0 = 0; j0 < cnt; j0 += EPW * UNROLL) {
            float4 r[UNROLL];
            float vv[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const int j = j0 + u * EPW + sub;
                const int32_t cj = __shfl_sync(0xffffffffu, c, j & 31);
                vv[u] = __shfl_sync(0xffffffffu, v, j & 31);
                if (j < cnt && active) {
                    r[u] = __ldg(reinterpret_cast<const float4 *>(x + (int64_t)cj * ldx) + fl);
                } else {
                    r[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    vv[u] = 0.f;
                }
            }
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                acc.x = fmaf(vv[u], r[u].x, acc.x);
                acc.y = fmaf(vv[u], r[u].y, acc.y);
                acc.z = fmaf(vv[u], r[u].z, acc.z);
                acc.w = fmaf(vv[u], r[u].w, acc.w);
            }
        }
    }
    // combine the EPW partial rows
#pragma unroll
    for (int o = LPR; o < 32; o <<= 1) {
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o);
        acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
        acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o);
        acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
    }
    if (sub == 0 && active) {
        if (bias) {
            const float4 bb = __ldg(reinterpret_cast<const float4 *>(bias) + fl);
            acc.x += bb.x; acc.y += bb.y; acc.z += bb.z; acc.w += bb.w;
        }
        if (act == PANGNN_ACT_ELU) {
            acc.x = elu1(acc.x); acc.y = elu1(acc.y); acc.z = elu1(acc.z); acc.w = elu1(acc.w);
        }
        reinterpret_cast<float4 *>(y + row * ldy)[fl] = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// Streaming variant for F in {32, 64, 128} (the widths the model uses).  The warp-per-row kernel
// above is latency-bound (ncu: no pipe above 40 %, 3 dependent memory round trips per row —
// rowptr -> (col, val) -> gathered rows — and a drained pipeline at every row boundary).  Here a
// warp owns a CHUNK of 32 consecutive rows: one coalesced rowptr load gives it the chunk's edge
// range, which is contiguous, so (col, val) are streamed 32 at a time with the next batch
// prefetched, and the gathers are issued UNROLL deep straight across row boundaries.  Rows are
// closed in order (warp-uniform test against the row end held by lane `cur`), so the sum order
// inside a row is the edge order — deterministic, no atomics.  A lane owns VEC = F/32 floats of
// the row (one 4/8/16-byte load per gathered row).
// ------------------------------------------------------------------------------------------------
template <int VEC> struct RowVec;
template <> struct RowVec<1> { using T = float; };
template <> struct RowVec<2> { using T = float2; };
template <> struct RowVec<4> { using T = float4; };

template <int VEC>
__device__ __forceinline__ void rv_load(float (&r)[VEC], const float *p) {
    const typename RowVec<VEC>::T t = __ldg(reinterpret_cast<const typename RowVec<VEC>::T *>(p));
    if constexpr (VEC == 1) { r[0] = t; }
    else if constexpr (VEC == 2) { r[0] = t.x; r[1] = t.y; }
    else { r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w; }
}

template <int VEC>
__device__ __forceinline__ void rv_store(float *p, const float (&r)[VEC]) {
    if constexpr (VEC == 1) { *p = r[0]; }
    else if constexpr (VEC == 2) { *reinterpret_cast<float2 *>(p) = make_float2(r[0], r[1]); }
    else { *reinterpret_cast<float4 *>(p) = make_float4(r[0], r[1], r[2], r[3]); }
}

constexpr int kRowsPerWarp = 32;

// IDENT: col == identity and val == ones (the CSR's entries ARE consecutive rows of x): the sorted-segment sum of
// per-edge rows that already lie in segment order (the scorer's da1 by source) — no (col, val) stream, row addresses
// known up front, so the gathers run UNROLL deep without the shuffle broadcast.
template <int VEC, int UNROLL, int MINB, bool IDENT = false>
__global__ void __launch_bounds__(256, MINB)
gcn_aggregate_stream_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                            const float *__restrict__ val, const float *__restrict__ x, int32_t ldx,
                            int32_t num_rows, const float *__restrict__ bias, int act,
                            float *__restrict__ y, int32_t ldy) {
    const int lane = threadIdx.x & 31;
    const int64_t r0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * kRowsPerWarp;
    if (r0 >= num_rows) return;
    const int nrows = (int)min((int64_t)kRowsPerWarp, (int64_t)num_rows - r0);
    // lane i holds the end of row r0 + i RELATIVE to the chunk's first edge (a chunk of 32 rows
    // never holds 2^31 edges); the chunk's edges are [0, n_edges) after rebasing col / val.
    const int64_t e_begin = rowptr[r0];
    const int my_end = (int)(rowptr[r0 + min(lane, nrows - 1) + 1] - e_begin);
    const int n_edges = __shfl_sync(0xffffffffu, my_end, nrows - 1);
    if (!IDENT) col += e_begin;
    if (!IDENT && val) val += e_begin;
    x += lane * VEC;
    if (IDENT) x += e_begin * (int64_t)ldx;
    y += r0 * (int64_t)ldy + lane * VEC;
    if (bias) bias += lane * VEC;

    int cur = 0;
    int cur_end = __shfl_sync(0xffffffffu, my_end, 0);
    float acc[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] = 0.f;

    auto close_row = [&]() {
        float o[VEC];
#pragma unroll
        for (int k = 0; k < VEC; ++k) o[k] = 0.f;
        if (bias) rv_load<VEC>(o, bias);                      // L1-resident after the first row
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            o[k] += acc[k];
            if (act == PANGNN_ACT_ELU) o[k] = elu1(o[k]);
            acc[k] = 0.f;
        }
        rv_store<VEC>(y + (int64_t)cur * ldy, o);
        ++cur;
        cur_end = __shfl_sync(0xffffffffu, my_end, cur & 31);
    };

    int32_t c_nxt = 0;
    float v_nxt = 0.f;
    if (!IDENT && lane < n_edges) {
        c_nxt = col[lane];
        v_nxt = val ? val[lane] : 1.0f;
    }
    for (int base = 0; base < n_edges; base += 32) {
        const int32_t c = c_nxt;
        const float v = v_nxt;
        const int nb = base + 32 + lane;
        if (!IDENT && nb < n_edges) {                         // prefetch the next 32 (col, val) pairs
            c_nxt = col[nb];
            v_nxt = val ? val[nb] : 1.0f;
        }
        const int cnt = min(32, n_edges - base);
        for (int j0 = 0; j0 < cnt; j0 += UNROLL) {
            float r[UNROLL][VEC];
            float vv[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const int j = j0 + u;
                const int32_t cj = IDENT ? base + j : __shfl_sync(0xffffffffu, c, j & 31);
                vv[u] = IDENT ? 1.0f : __shfl_sync(0xffffffffu, v, j & 31);
                if (j < cnt) {
                    rv_load<VEC>(r[u], x + (int64_t)cj * ldx);
                } else {
#pragma unroll
                    for (int k = 0; k < VEC; ++k) r[u][k] = 0.f;
                }
            }
            const int e0 = base + j0;
            if (e0 + UNROLL <= cur_end) {                     // whole group inside the open row
#pragma unroll
                for (int u = 0; u < UNROLL; ++u)
#pragma unroll
                    for (int k = 0; k < VEC; ++k) acc[k] = fmaf(vv[u], r[u][k], acc[k]);
            } else {
#pragma unroll
                for (int u = 0; u < UNROLL; ++u) {
                    if (e0 + u < n_edges) {                   // warp-uniform
                        while (e0 + u >= cur_end) close_row();    // rows ending before this edge (incl. empty ones)
#pragma unroll
                        for (int k = 0; k < VEC; ++k) acc[k] = fmaf(vv[u], r[u][k], acc[k]);
                    }
                }
            }
        }
    }
    while (cur < nrows) close_row();                          // last row and trailing empty rows
}

// Wide rows (F > 128): one warp per row, loop over 128-float column panels.
__global__ void __launch_bounds__(256)
gcn_aggregate_wide_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                          const float *__restrict__ val, const float *__restrict__ x, int64_t ldx,
                          int32_t num_rows, int32_t feat, const float *__restrict__ bias, int act,
                          float *__restrict__ y, int64_t ldy) {
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= num_rows) return;
    const int64_t b = rowptr[row], e = rowptr[row + 1];
    for (int f0 = 0; f0 < feat; f0 += 128) {
        const bool active = f0 + lane * 4 < feat;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int64_t i = b; i < e; ++i) {
            const float v = val ? val[i] : 1.0f;
            if (active) {
                const float4 r = __ldg(reinterpret_cast<const float4 *>(x + (int64_t)col[i] * ldx + f0) + lane);
                acc.x = fmaf(v, r.x, acc.x); acc.y = fmaf(v, r.y, acc.y);
                acc.z = fmaf(v, r.z, acc.z); acc.w = fmaf(v, r.w, acc.w);
            }
        }
        if (active) {
            if (bias) {
                const float4 bb = __ldg(reinterpret_cast<const float4 *>(bias + f0) + lane);
                acc.x += bb.x; acc.y += bb.y; acc.z += bb.z; acc.w += bb.w;
            }
            if (act == PANGNN_ACT_ELU) {
                acc.x = elu1(acc.x); acc.y = elu1(acc.y); acc.z = elu1(acc.z); acc.w = elu1(acc.w);
            }
            reinterpret_cast<float4 *>(y + row * ldy + f0)[lane] = acc;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// activation backward + bias gradient
// ------------------------------------------------------------------------------------------------
constexpr int kActRowsPerChunk = 64;
constexpr int kActMaxBlocks = kNumSMs * 8;      // persistent: <= 1184 per-block partial rows

// Block (feat/4 x TY threads) walks 64-row chunks grid-stride; each thread keeps a float4 column sum.
__global__ void __launch_bounds__(256)
act_bwd_bias_kernel(const float *__restrict__ dy, const float *__restrict__ yv, int64_t num_rows,
                    int32_t feat, int act, float *__restrict__ g, float *__restrict__ partial) {
    extern __shared__ float4 red[];                        // [TY][feat/4]
    const int fq = feat / 4;
    const int tx = threadIdx.x % fq, ty = threadIdx.x / fq;
    const int TY = blockDim.x / fq;
    const int64_t nchunks = (num_rows + kActRowsPerChunk - 1) / kActRowsPerChunk;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ty < TY) {
        for (int64_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
            const int64_t r0 = chunk * kActRowsPerChunk;
            const int64_t r1 = min(r0 + (int64_t)kActRowsPerChunk, num_rows);
            for (int64_t r = r0 + ty; r < r1; r += TY) {
                float4 d = ld_stream_f4(dy + r * feat + tx * 4);
                if (act == PANGNN_ACT_ELU) {
                    const float4 o = ld_stream_f4(yv + r * feat + tx * 4);
                    d.x *= o.x > 0.f ? 1.f : o.x + 1.f;
                    d.y *= o.y > 0.f ? 1.f : o.y + 1.f;
                    d.z *= o.z > 0.f ? 1.f : o.z + 1.f;
                    d.w *= o.w > 0.f ? 1.f : o.w + 1.f;
                }
                if (g) reinterpret_cast<float4 *>(g + r * feat)[tx] = d;
                s.x += d.x; s.y += d.y; s.z += d.z; s.w += d.w;
            }
        }
        red[ty * fq + tx] = s;
    }
    __syncthreads();
    if (ty == 0) {
        for (int t = 1; t < TY; ++t) {
            const float4 o = red[t * fq + tx];
            s.x += o.x; s.y += o.y; s.z += o.z; s.w += o.w;
        }
        reinterpret_cast<float4 *>(partial + (int64_t)blockIdx.x * feat)[tx] = s;
    }
}

// Deterministic second stage: out[c] = sum_b partial[b][c] (fp64 accumulate, fixed order).
__global__ void __launch_bounds__(256)
reduce_partials_kernel(const float *__restrict__ partial, int64_t nblocks, int32_t width,
                       int32_t stride, float *__restrict__ out) {
    __shared__ double red[8][33];
    const int c = blockIdx.x * 32 + (threadIdx.x & 31);
    const int slice = threadIdx.x >> 5;                    // 8 slices of the block range
    double s = 0.0;
    if (c < width)
        for (int64_t b = slice; b < nblocks; b += 8) s += (double)partial[b * stride + c];
    red[slice][threadIdx.x & 31] = s;
    __syncthreads();
    if (slice == 0 && c < width) {
        double t = 0.0;
        for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x & 31];
        out[c] = (float)t;
    }
}

int reduce_partials(const float *partial, int64_t nblocks, int32_t width, int32_t stride, float *out,
                    cudaStream_t st) {
    reduce_partials_kernel<<<(width + 31) / 32, 256, 0, st>>>(partial, nblocks, width, stride, out);
    PANGNN_CHECK_LAUNCH("reduce_partials");
    return PANGNN_OK;
}

}  // namespace pangnn

using namespace pangnn;

extern "C" {

int pangnn_gcn_norm(const int64_t *rowptr, const int32_t *col, const uint32_t *perm, const float *w,
                    int32_t N, float *dis, float *val, void *stream) {
    PANGNN_REQUIRE(rowptr && dis && N >= 0, "null pointer");
    if (N == 0) return PANGNN_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)(((int64_t)N * 32 + 255) / 256);
    gcn_deg_kernel<<<blocks, 256, 0, st>>>(rowptr, perm, w, N, dis);
    PANGNN_CHECK_LAUNCH("gcn_deg");
    if (val) {
        gcn_val_kernel<<<blocks, 256, 0, st>>>(rowptr, col, perm, w, dis, N, 1, val);
        PANGNN_CHECK_LAUNCH("gcn_val");
    }
    return PANGNN_OK;
}

int pangnn_gcn_norm_apply(const int64_t *rowptr, const int32_t *col, const uint32_t *perm,
                          const float *w, const float *dis, int32_t N, int rows_are_dst, float *val,
                          void *stream) {
    PANGNN_REQUIRE(rowptr && dis, "null pointer");   // col/val/perm may be NULL for an edgeless graph
    if (N == 0) return PANGNN_OK;
    const unsigned blocks = (unsigned)(((int64_t)N * 32 + 255) / 256);
    gcn_val_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rowptr, col, perm, w, dis, N,
                                                            rows_are_dst, val);
    PANGNN_CHECK_LAUNCH("gcn_val");
    return PANGNN_OK;
}

int pangnn_gcn_aggregate(const int64_t *rowptr, const int32_t *col, const float *val, const float *x,
                         int64_t ldx, int32_t num_rows, int32_t feat, const float *bias, int act,
                         float *y, int64_t ldy, void *stream) {
    if (num_rows == 0) return PANGNN_OK;
    PANGNN_REQUIRE(rowptr && y, "null pointer");       // x may be NULL when the graph has no edge
    PANGNN_REQUIRE(col || (!val && (feat == 32 || feat == 64 || feat == 128) && ldx < (1 << 30) && ldy < (1 << 30)),
                   "col == NULL (identity: entry i of the CSR is row i of x) needs val == NULL and feat in {32, 64, 128}");
    PANGNN_REQUIRE(feat > 0 && feat % 4 == 0 && feat <= 512, "feat must be a multiple of 4, <= 512");
    PANGNN_REQUIRE(ldx % 4 == 0 && ldy % 4 == 0 && ldx >= feat && ldy >= feat, "bad row stride");
    PANGNN_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)y % 16 == 0) &&
                       (!bias || (uintptr_t)bias % 16 == 0), "pointers must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)(((int64_t)num_rows * 32 + 255) / 256);
#define LAUNCH(LPR, UNR)                                                                          \
    gcn_aggregate_kernel<LPR, UNR><<<blocks, 256, 0, st>>>(rowptr, col, val, x, ldx, num_rows,    \
                                                           feat, bias, act, y, ldy)
    if ((feat == 32 || feat == 64 || feat == 128) && ldx < (1 << 30) && ldy < (1 << 30)) {
        // (UNROLL, min CTAs/SM) from a sweep on B200 over the C3 union graph (tools/tune_agg.py):
        // 4 gathers in flight per warp and as many resident warps as the register file allows
        // beat deeper unrolling at lower occupancy (F=128: 1.09 ms vs 1.36 ms at UNROLL 8,
        // 3.4 ms at UNROLL 16; warp-per-row kernel 1.77 ms).
        const int64_t warps = ((int64_t)num_rows + kRowsPerWarp - 1) / kRowsPerWarp;
        const unsigned sblocks = (unsigned)((warps * 32 + 255) / 256);
#define SLAUNCH(VEC, UNR, MINB)                                                                   \
    gcn_aggregate_stream_kernel<VEC, UNR, MINB><<<sblocks, 256, 0, st>>>(                         \
        rowptr, col, val, x, (int32_t)ldx, num_rows, bias, act, y, (int32_t)ldy)
        if (!col) {                                             // identity columns (PANGNN_REQUIRE above: val == NULL too)
            if (feat == 128) gcn_aggregate_stream_kernel<4, 8, 3, true><<<sblocks, 256, 0, st>>>(
                rowptr, nullptr, nullptr, x, (int32_t)ldx, num_rows, bias, act, y, (int32_t)ldy);
            else if (feat == 64) gcn_aggregate_stream_kernel<2, 8, 4, true><<<sblocks, 256, 0, st>>>(
                rowptr, nullptr, nullptr, x, (int32_t)ldx, num_rows, bias, act, y, (int32_t)ldy);
            else gcn_aggregate_stream_kernel<1, 8, 4, true><<<sblocks, 256, 0, st>>>(
                rowptr, nullptr, nullptr, x, (int32_t)ldx, num_rows, bias, act, y, (int32_t)ldy);
        } else if (feat == 128) SLAUNCH(4, 4, 4);
        else if (feat == 64) SLAUNCH(2, 4, 6);
        else SLAUNCH(1, 4, 6);
#undef SLAUNCH
    } else if (feat <= 16) LAUNCH(4, 2);
    else if (feat <= 32) LAUNCH(8, 2);
    else if (feat <= 64) LAUNCH(16, 4);
    else if (feat <= 128) LAUNCH(32, 8);
    else
        gcn_aggregate_wide_kernel<<<blocks, 256, 0, st>>>(rowptr, col, val, x, ldx, num_rows, feat,
                                                          bias, act, y, ldy);
#undef LAUNCH
    PANGNN_CHECK_LAUNCH("gcn_aggregate");
    return PANGNN_OK;
}

static int64_t act_blocks(int64_t num_rows) {
    const int64_t nchunks = (num_rows + kActRowsPerChunk - 1) / kActRowsPerChunk;
    return nchunks < 1 ? 1 : (nchunks < kActMaxBlocks ? nchunks : kActMaxBlocks);
}

size_t pangnn_act_bwd_bias_workspace_bytes(int64_t num_rows, int32_t feat) {
    return (size_t)act_blocks(num_rows) * feat * sizeof(float) + 256;
}

int pangnn_act_bwd_bias(const float *dy, const float *yv, int64_t num_rows, int32_t feat, int act,
                        float *g, float *dbias, void *ws, size_t ws_bytes, void *stream) {
    PANGNN_REQUIRE(dbias && ws, "null pointer");
    PANGNN_REQUIRE(feat > 0 && feat % 4 == 0 && feat <= 1024, "feat must be a multiple of 4, <= 1024");
    if (ws_bytes < pangnn_act_bwd_bias_workspace_bytes(num_rows, feat)) {
        set_error("act_bwd_bias: workspace too small");
        return PANGNN_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // zero rows: the inputs are empty tensors, whose data pointer is NULL
    if (num_rows == 0) return check_cuda(cudaMemsetAsync(dbias, 0, feat * sizeof(float), st), "memset");
    PANGNN_REQUIRE(dy, "null pointer");
    PANGNN_REQUIRE(act == PANGNN_ACT_NONE || yv, "activation output required");
    const int64_t nb = act_blocks(num_rows);
    const int fq = feat / 4;
    const int TY = 256 / fq;
    float *partial = static_cast<float *>(ws);
    act_bwd_bias_kernel<<<(unsigned)nb, 256, (size_t)TY * fq * sizeof(float4), st>>>(
        dy, yv, num_rows, feat, act, g, partial);
    PANGNN_CHECK_LAUNCH("act_bwd_bias");
    return reduce_partials(partial, nb, feat, feat, dbias, st);
}

}  // extern "C"
